/* raxtax_host.h -- C ABI of the C++ host library (libraxtax_host.so) that sits above include/raxtax_b200.h.
 *
 * The reference's host is Rust; no Rust toolchain exists in the build image, so the host side of the hot path
 * is C++17 with the same names, argument meaning and error behaviour as the reference:
 *   rxh_tree_from_fasta   = parser::parse_reference_fasta_str   (src/parser.rs:46-105) -> Tree::new (src/tree.rs:47-140)
 *   rxh_tree_new          = Tree::new                            (src/tree.rs:47-140)
 *   rxh_queries_from_fasta= parser::parse_query_fasta_str        (src/parser.rs:117-154)
 *   rxh_raxtax            = raxtax::raxtax                       (src/raxtax.rs:14-97)
 *   rxh_sender            = crossbeam Sender<(String,String,Option<String>)> (src/raxtax.rs:20, src/main.rs:126-134)
 * Functions returning int give 0 on success, negative on failure with the message in rxh_last_error();
 * constructors return NULL on failure.  Errors the reference reports with bail!/panic! surface as failures
 * with the same message text where one exists.
 */
#ifndef RAXTAX_HOST_H
#define RAXTAX_HOST_H

#include <stddef.h>
#include <stdint.h>

#include "raxtax_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rxh_tree rxh_tree;       /* raxtax::tree::Tree */
typedef struct rxh_queries rxh_queries; /* Vec<(String, Vec<u8>)> */

const char* rxh_last_error(void);

/* ---- Tree ------------------------------------------------------------------------------------------------ */
rxh_tree* rxh_tree_from_fasta(const char* text, size_t len);
/* lineages: n strings joined by '\n'; sequences: 4-bit codes (parser.rs:11-34) with offsets[n+1] */
rxh_tree* rxh_tree_new(size_t n, const char* lineage_blob, size_t blob_len, const uint64_t* seq_offsets, const uint8_t* seq_codes);
/* Binary database (bincode 1.3 image of Tree; tree.rs:146-164, layout in SURVEY.md Appendix C).
 * rxh_tree_from_bin = Tree::load_from_file: NULL when the bytes do not deserialise (the caller then parses them as FASTA, as
 * parser::parse_reference_fasta_file does, parser.rs:37-44); a loaded tree carries its k_mer_map, which is then what the
 * device index is built from.  rxh_tree_save_bin = Tree::save_to_file.  32-bit ids only (not the `huge_db` feature). */
rxh_tree* rxh_tree_from_bin(const void* data, size_t len);
/* parser::parse_reference_fasta_file (parser.rs:37-44): the file is loaded as a binary database if it deserialises as one
 * (*was_database = 1), else parsed as FASTA, plain or gz -- in blocks that are read / decompressed on one thread while the previous
 * block is parsed on all the others, so that the text is never held in memory as a whole.  rxh_queries_from_file likewise
 * (parser.rs:108-115, without the skip filter: rxh_queries_skip). */
rxh_tree* rxh_tree_from_file(const char* path, int* was_database);
int rxh_tree_save_bin(const rxh_tree* t, const char* path);
void rxh_tree_free(rxh_tree* t);
size_t rxh_tree_num_tips(const rxh_tree* t);
const char* rxh_tree_lineage(const rxh_tree* t, size_t i); /* Tree.lineages[i] (sorted order) */
/* Tree.k_mer_map as CSR (pointers stay valid for the life of the tree) */
/* Tree.k_mer_map (tree.rs:41) is materialised on first use only: the device builds its index from the sorted sequences
 * (rtx_index_desc.ref_seq_*), so classification never needs the lists on the host.  rxh_tree_build_kmer_map forces it (after which
 * rxh_tree_index_desc / rxh_tree_upload hand the CSR to the device instead); rxh_tree_csr builds it if needed and returns it. */
void rxh_tree_build_kmer_map(const rxh_tree* t);
int rxh_tree_has_kmer_map(const rxh_tree* t);
void rxh_tree_csr(const rxh_tree* t, const uint64_t** offsets, const uint32_t** ids);
/* Tree.sequences.get(seq): number of matches; up to cap ascending ids are written */
size_t rxh_tree_exact(const rxh_tree* t, const uint8_t* seq, size_t len, uint32_t* out, size_t cap);
/* flattened Inner/Taxon node arrays + everything rtx_index_upload needs; pointers owned by the tree */
int rxh_tree_index_desc(const rxh_tree* t, rtx_index_desc* out);
/* convenience: rtx_index_upload(ctx, desc of t) restricted to references [shard_begin, shard_end) (0,0 = all) */
int rxh_tree_upload(const rxh_tree* t, rtx_ctx* ctx, uint64_t shard_begin, uint64_t shard_end);
/* reference-sharded upload: this context becomes shard `shard_rank` of `n_shards` (rtx_index_desc.shard_cuts) */
int rxh_tree_upload_sharded(const rxh_tree* t, rtx_ctx* ctx, uint32_t n_shards, uint32_t shard_rank, const uint64_t* shard_cuts);

/* ---- queries ----------------------------------------------------------------------------------------------- */
rxh_queries* rxh_queries_from_fasta(const char* text, size_t len);
rxh_queries* rxh_queries_from_file(const char* path);
rxh_queries* rxh_queries_new(size_t n, const char* label_blob, size_t blob_len, const uint64_t* seq_offsets, const uint8_t* seq_codes);
/* drop the queries whose label is listed ('\n'-separated, the content of raxtax.ckp): parse_query_fasta_str's queries_to_skip
 * filter (parser.rs:108-115,150-153) */
int rxh_queries_skip(rxh_queries* q, const char* label_blob, size_t blob_len);
void rxh_queries_free(rxh_queries* q);
size_t rxh_queries_len(const rxh_queries* q);
const char* rxh_queries_label(const rxh_queries* q, size_t i);
void rxh_queries_arrays(const rxh_queries* q, const uint64_t** seq_offsets, const uint8_t** seq_codes);

/* ---- driver ------------------------------------------------------------------------------------------------
 * sender(user, query_label, primary_results, tsv_results_or_NULL) is called once per query, in query order,
 * from the calling thread (rxh_raxtax; see rxh_raxtax_multi for several GPUs); a non-zero return aborts the run like a failed channel send (raxtax.rs:87).
 * logger(user, level, message) receives the Info / Warn lines the reference writes to raxtax.log
 * (raxtax.rs:46-52): level 2 = Warn, 3 = Info; it is called from the driver threads (serialised with the sender).
 * chunk_size = queries per device batch (0 = about an eighth of the queries per GPU, between 1024 and 32768).  The driver keeps
 * two batches in flight per GPU: while one runs, the next is prepared and uploaded and the previous one is formatted and sent,
 * so results (and a caller's progress file) appear chunk by chunk while the run is going.  A batch that does not fit the device
 * memory is split in halves and retried.
 * Returns 0, or -1 on error; *warnings (may be NULL) is set when exact matches disagreed above the leaf level
 * (raxtax.rs:49-52, 93-95).
 */
typedef int (*rxh_sender)(void* user, const char* query_label, const char* primary_results, const char* tsv_results);
typedef void (*rxh_logger)(void* user, int level, const char* message);

/* A sender / logger pair that only counts (queries, result lines, bytes, an order-independent checksum of the primary strings):
 * what a benchmark or a test hands to rxh_raxtax as the writer side of the channel.  user = rxh_counts*, zero-initialised by the caller. */
typedef struct {
    uint64_t queries, lines, label_bytes, primary_bytes, tsv_bytes, checksum, log_lines, log_bytes, warn_lines;
} rxh_counts;
int rxh_count_sender(void* user, const char* query_label, const char* primary_results, const char* tsv_results);
void rxh_count_logger(void* user, int level, const char* message);
/* `{:.N}` of an f64 as the result lines print confidences (N = 2) and signals (N = 5) (lineage.rs:17-30): the exact binary value
 * rounded to nearest, ties to even.  Exposed so that tests can pin the fast path against the C library's conversion. */
size_t rxh_format_fixed(double value, int precision, char* out, size_t cap);

/* The chunks rxh_raxtax / rxh_raxtax_multi cut a job of n_queries into for n_ctx contexts (the reference's par_chunks, raxtax.rs:35-39,
 * main.rs:119-124): chunk i = [begins[i], begins[i + 1]).  chunk_size 0 = the library's choice (about eight chunks per context, smaller
 * ones at both ends of the job so that the host work before the first launch and behind the last one is short).  Writes at most cap
 * values, returns how many there are.  Exposed for tests. */
size_t rxh_plan_chunks(size_t n_queries, size_t n_ctx, size_t chunk_size, size_t* begins, size_t cap);

int rxh_raxtax(rtx_ctx* ctx, const rxh_queries* queries, const rxh_tree* tree, int skip_exact_matches, int raw_confidence,
               size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger, void* logger_user, int* warnings);

/* The driver keeps its page-locked result buffers per context between calls (allocating them costs milliseconds and waits for the
 * device); this frees them.  Call it before rtx_ctx_destroy of a context that was used with rxh_raxtax if the process goes on. */
void rxh_release_buffers(void);

/* The same over several GPUs of one box (BASELINE config 3: queries partitioned, index replicated, no collective): ctxs[i] each hold
 * the whole index of `tree` (rxh_tree_upload); one driver thread per context pulls chunks of chunk_size queries (0 = ~8 chunks per
 * context, 1024..32768 queries) from a shared counter, as rayon's par_chunks does for the reference (raxtax.rs:35-39, main.rs:119-124).
 * sender / logger are serialised; queries arrive in completion order (the reference's channel gives no order either). */
int rxh_raxtax_multi(rtx_ctx* const* ctxs, size_t n_ctx, const rxh_queries* queries, const rxh_tree* tree, int skip_exact_matches,
                     int raw_confidence, size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger,
                     void* logger_user, int* warnings);

/* rxh_raxtax_multi with every query classified in the orientation that shares more 8-mers with some reference (--strand both,
 * RTX_BOTH_STRANDS in include/raxtax_b200.h): per distinct sequence the host also looks up the exact matches of its reverse complement;
 * the exact-match log lines and the "differ above the leafs" warning are those of the classified orientation (written once the
 * batch's strands are known); every line of the primary and the tsv string ends in a strand column (`\t+` as given, `\t-` reverse
 * complement) and the tsv line carries the sequence in the classified orientation.  Not available over a reference-sharded index. */
int rxh_raxtax_both_strands(rtx_ctx* const* ctxs, size_t n_ctx, const rxh_queries* queries, const rxh_tree* tree, int skip_exact_matches,
                            int raw_confidence, size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger,
                            void* logger_user, int* warnings);

/* rxh_raxtax_multi (both_strands = 0) or rxh_raxtax_both_strands (1) that also reports each query's best hits (RTX_OPT_BEST_HITS =
 * best_hits, 1..64; 0 = none and hits_sender is never called): hits_sender(hits_user, query_label, hit_lines) is called right before the
 * query's sender, on the same thread.  hit_lines holds one line per hit, '\n'-separated, without a final newline, empty for a query
 * without hits: `{label}\t{rank 1..}\t{lineage}\t{shared 8-mers}\t{K}\t{reference id}`, with both_strands followed by the strand column
 * (`\t+` / `\t-`).  Reference ids are positions in Tree.lineages.  Not available over a reference-sharded index. */
typedef int (*rxh_hits_sender)(void* user, const char* query_label, const char* hit_lines);
int rxh_raxtax_best_hits(rtx_ctx* const* ctxs, size_t n_ctx, const rxh_queries* queries, const rxh_tree* tree, int skip_exact_matches,
                         int raw_confidence, size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger,
                         void* logger_user, int* warnings, int both_strands, uint32_t best_hits, rxh_hits_sender hits_sender,
                         void* hits_user);

/* raxtax::raxtax over a reference-sharded index (BASELINE config 5: databases too large to replicate) with all shards driven by this
 * process: ctxs[r] holds shard r of n_ctx (rxh_tree_upload_sharded).  When every shard sits on its own GPU the contexts are joined into
 * an NCCL communicator and one driver thread per rank calls rtx_shard_run / rtx_shard_gather (histogram all-reduce, record all-gather
 * and the gather + merge of the result lines all inside the device library); rank 0's lines feed the same writer side as rxh_raxtax.
 * Several shards on one GPU (NCCL does not take two ranks on one device; RXH_SHARD_NO_NCCL=1 forces this path): phase by phase with the
 * exchanges staged through pinned host memory and the merge on the host.  Lines are sent in query order from the calling thread.
 * chunk_size = queries per sharded batch (0 = a quarter of the queries, 2048..32768, over NCCL; up to 8192 on the staged path, halved
 * automatically until a batch fits one sub-batch of every shard). */
int rxh_raxtax_sharded(rtx_ctx* const* ctxs, size_t n_ctx, const rxh_queries* queries, const rxh_tree* tree, int skip_exact_matches,
                       int raw_confidence, size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger,
                       void* logger_user, int* warnings);

/* Reference-sharded mode (BASELINE config 5): merge of the result lines the ranks emitted for one batch -- per query the ranks' lines
 * in the order of lineage.rs:93, then the one-exact-match override of raxtax.rs:73-84 (which needs the best line of all ranks).
 * Inputs are the rtx_results arrays of every rank (confidence rows have max_levels entries); the caller sizes the outputs for the
 * sum of the ranks' line counts.  Returns 0, or -1 (rxh_last_error) e.g. for a query without any line (raxtax.rs:72). */
int rxh_merge_shard_results(size_t n_ranks, size_t n_queries, uint32_t max_levels, const uint32_t* const* result_begin,
                            const uint32_t* const* first_ref, const uint8_t* const* n_levels, const double* const* confidence,
                            const double* const* local_signal, const uint32_t* exact_offsets, const uint32_t* exact_ids,
                            const uint8_t* ref_levels, int skip_exact_matches, int raw_confidence, uint32_t* out_begin, uint32_t* out_first,
                            uint8_t* out_nlev, double* out_conf, double* out_local, uint64_t out_capacity, uint64_t* n_out);

/* exact-match lookup for a whole batch (the host half of raxtax.rs:42): fills exact_offsets[n+1]; returns the
 * total number of ids; writes at most cap ids */
uint64_t rxh_exact_batch(const rxh_tree* t, size_t n, const uint64_t* seq_offsets, const uint8_t* seq_codes, uint32_t* exact_offsets,
                         uint32_t* exact_ids, uint64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* RAXTAX_HOST_H */
