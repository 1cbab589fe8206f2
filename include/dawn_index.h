/*
 * dawn_index.h -- C ABI of libdawn_b200.so: a device-resident exact top-k index for
 * 384-d page embeddings on NVIDIA B200 (sm_100a).
 *
 * Drop-in boundary: these entry points are what a Rust FFI layer binds in place of the
 * `usearch::ffi` cxx bridge that the reference uses today.  Each function names the
 * reference interface it replaces (paths relative to dawn-search/dawnsearch v0.2.0):
 *
 *   reference (usearch::ffi, called from src/search/search_provider.rs)      this header
 *   ---------------------------------------------------------------------   ----------------------
 *   new_index(&IndexOptions)              :35-42, :102                       dawn_index_create
 *   drop(UniquePtr<Index>)                :67                                dawn_index_free
 *   Index::reserve(usize)                 :133, :282                         dawn_index_reserve
 *   Index::add(u64, &[f32])               :149, :284                         dawn_index_add / _add_batch
 *   Index::search(&[f32], usize)->Matches :214, :221                         dawn_index_search / _search_batch
 *   Index::size() / capacity()            :246, :280                         dawn_index_size / _capacity
 *   Index::dimensions()                   (IndexOptions.dimensions :36)      dawn_index_dimensions
 *   Index::save(&str) / load(&str)        :115, :117, :178                   dawn_index_save / _load
 *   Index::view(&str)  (examples_old/search_usearch.rs:47)                   dawn_index_load
 *   cxx::Exception -> Result::Err         :102,:117,:133,:149,:214,:284      negative return + dawn_last_error()
 *
 * Semantics kept from the reference: distances are "smaller is better" and equal
 * 1 - dot(query, stored) (src/search/vector.rs:128-134; consumers: src/net/web.rs:330-343,
 * src/net/udp_service.rs:196-199, src/search/best_results.rs:56); results come back
 * ascending by distance; labels are caller-supplied u64 page ids (SQLite rowids); fewer
 * than k results are returned when the index holds fewer than k vectors; the caller checks
 * that vectors are L2-normalised before calling (search_provider.rs:206,265).
 * Added on top: the search is exact (not HNSW) over the stored fp16 vectors and ties break
 * deterministically on the lower label.
 *
 * There is NO CPU fallback: every call that needs the GPU fails with DAWN_ERR_CUDA if no
 * sm_100 device is usable.
 *
 * Threading: the reference drives its index from a single thread
 * (src/bin/dawnsearch.rs:76-78); that model works unchanged.  Beyond it, search* / get are re-entrant:
 * every host search leases its own stream + workspace (up to 8 in flight per handle), so several threads
 * may search one handle concurrently.  add* / remove* / reserve / save / load are serialised among themselves; an
 * add never waits for running searches (it appends beyond what they see), only a reallocation or a remove does.
 * A handle may be used from any thread; different handles are independent.
 */
#ifndef DAWN_INDEX_H
#define DAWN_INDEX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DAWN_DIMENSIONS 384 /* src/search/vector.rs:26 EM_LEN */
#define DAWN_MAX_K 120      /* largest k one search call accepts */

enum {
    DAWN_OK = 0,
    DAWN_ERR_INVALID = -1,   /* bad argument (null pointer, k out of range, wrong dimension) */
    DAWN_ERR_CUDA = -2,      /* CUDA failure; sticky: the handle refuses further work */
    DAWN_ERR_CAPACITY = -3,  /* add beyond reserved capacity (usearch raises the same way) */
    DAWN_ERR_IO = -4,        /* save / load failed; the index is unchanged */
    DAWN_ERR_INTERNAL = -5
};

/* usearch ScalarKind equivalents for the stored corpus (search_provider.rs:38). */
enum {
    DAWN_SCALAR_F16 = 0, /* fp16 rows, 768 B per vector: "exact" = exact over the fp16-rounded vectors */
    DAWN_SCALAR_I8 = 1,  /* int8 + per-vector f32 scale, 388 B per vector */
    DAWN_SCALAR_F32 = 2  /* the reference's own ScalarKind::F32 (search_provider.rs:38): the f32 vectors are kept as given
                          * (1536 B) beside an fp16 selection copy (768 B); distances are those of an exact f32 brute force
                          * over the vectors as added, bit for bit */
};
/* usearch MetricKind::IP (search_provider.rs:37) is the only metric the reference uses. */
enum { DAWN_METRIC_IP = 0 };

typedef struct dawn_options {
    uint32_t dimensions; /* must be 384 (0 = default) */
    uint32_t metric;     /* DAWN_METRIC_IP */
    uint32_t scalar;     /* DAWN_SCALAR_F16, DAWN_SCALAR_I8 (per-vector absmax/127 scale) or DAWN_SCALAR_F32 */
    int32_t device;      /* CUDA device ordinal */
    uint64_t capacity;   /* vectors to reserve up front (0 = none) */
    uint32_t flags;      /* reserved, 0 */
    uint32_t reserved_;
} dawn_options;

typedef struct dawn_index dawn_index;

/* Per-thread message for the last failing call on this thread ("" if none). */
const char *dawn_last_error(void);
/* "libdawn_b200 <version> sm_100a" */
const char *dawn_version(void);

int dawn_index_create(const dawn_options *opts, dawn_index **out);
void dawn_index_free(dawn_index *idx);

/* Grow capacity to at least n vectors (never shrinks).  Existing vectors are kept. */
int dawn_index_reserve(dawn_index *idx, size_t n);
/* Append one / n labelled f32 vectors (host memory).  Vectors become visible to the next
 * search.  Fails with DAWN_ERR_CAPACITY when size + n > capacity (the reference grows by
 * reserve(size+1024) itself, search_provider.rs:280-283). */
int dawn_index_add(dawn_index *idx, uint64_t label, const float *vector384);
int dawn_index_add_batch(dawn_index *idx, const uint64_t *labels, const float *vectors, size_t n);
/* Remove every stored row whose label is in labels[0..n) (duplicates in the list and absent labels are fine).
 * *removed_out (may be NULL) = rows removed.  Staged adds made before the call are covered.  size() drops by the
 * count; capacity is unchanged.  Like a reallocation, it waits for searches in flight; searches that start later
 * see the new corpus.  Serialised with add* / reserve / save / load.  The last rows of the corpus move into the
 * freed places (exact search does not depend on row order).  An update is a remove followed by an add.
 * n > 0 with labels == NULL, or a NULL handle: DAWN_ERR_INVALID. */
int dawn_index_remove_batch(dawn_index *idx, const uint64_t *labels, size_t n, size_t *removed_out);
int dawn_index_remove(dawn_index *idx, uint64_t label, size_t *removed_out);

/* Exact top-k for one / `batch` f32 queries in host memory.  Output buffers are caller
 * allocated: labels[batch*k], distances[batch*k], counts[batch]; row b's results occupy
 * [b*k, b*k + counts[b]), ascending by distance, ties by ascending label. */
int dawn_index_search(dawn_index *idx, const float *query384, size_t k, uint64_t *labels_out,
                      float *distances_out, size_t *count_out);
int dawn_index_search_batch(dawn_index *idx, const float *queries, size_t batch, size_t k,
                            uint64_t *labels_out, float *distances_out, size_t *counts_out);

size_t dawn_index_size(const dawn_index *idx);
size_t dawn_index_capacity(const dawn_index *idx);
size_t dawn_index_dimensions(const dawn_index *idx);

/* Persist / restore the stored corpus (rows as stored: f32 / fp16 / int8+scale, and labels) at `path`.
 * load: an EMPTY index whose reserved capacity covers the file (the start-up sequence reserve -> load) is filled in
 * place, so a 100M-row shard never needs two arenas; a non-empty index gets a fresh arena that is swapped in only when
 * the whole file has arrived (a failed load then leaves the index unchanged). */
int dawn_index_save(dawn_index *idx, const char *path);
int dawn_index_load(dawn_index *idx, const char *path);

/* Stored vector for `label` decoded to f32 (SearchProvider::embedding_for_page,
 * search_provider.rs:183-195, served from the device corpus).  DAWN_ERR_INVALID if absent. */
int dawn_index_get(dawn_index *idx, uint64_t label, float *vector384_out);

/* SearchProvider::verify (search_provider.rs:289-327) over the device corpus: one HBM-bound pass that applies
 * the reference's gate (finite, 0.99 < |v| < 1.01; src/search/vector.rs:185-192) to every STORED row.  The
 * blob-length check of the reference is structural here.  Any pointer may be NULL.  The library runs the same
 * pass incrementally over newly added rows before a search: if a stored row is longer than the gate allows,
 * every bound of the exactness certificate is scaled accordingly (the raw ABI, like usearch, accepts any vector). */
int dawn_index_verify(dawn_index *idx, size_t *bad_rows_out, float *min_norm_out, float *max_norm_out);

/* ---- device-resident entry points (no host<->device copies inside the call) -------------
 * For callers that already hold queries / want results in device memory (a batching
 * front-end, the multi-GPU merge, bench.py's kernel-only timing).  `stream` is a
 * cudaStream_t passed as void* (NULL = the index's own stream); the call only enqueues.
 * counts_out / flags_out are uint32 per query; flags bit0 = exactness certified. */
int dawn_index_search_device(dawn_index *idx, const float *d_queries, size_t batch, size_t k,
                             uint64_t *d_labels_out, float *d_distances_out,
                             uint32_t *d_counts_out, uint32_t *d_flags_out, void *stream);
/* The same with UdpPacket::Search's distance_limit (NaN = none): pushed down into the kernels' thresholds, and
 * the counts are cut on the device so that only hits with distance < limit remain (results ascend). */
int dawn_index_search_device_limit(dawn_index *idx, const float *d_queries, size_t batch, size_t k, float distance_limit,
                                   uint64_t *d_labels_out, float *d_distances_out,
                                   uint32_t *d_counts_out, uint32_t *d_flags_out, void *stream);
/* Merge `n_lists` per-shard result lists (each [batch][k] labels + distances, ascending,
 * with [batch] counts) into one [batch][k] list; the device-side step after the all-gather of
 * a sharded search (the role of search_remote's BestResults merge,
 * src/search/search_service.rs:247-268).  List l's three arrays start l*list_stride_bytes
 * after the three base pointers, so one packed block per shard (as it lands from a single
 * all-gather) can be merged in place; list_stride_bytes == 0 means three dense arrays
 * [n_lists][batch][k] / [n_lists][batch].  n_lists <= 64 and n_lists*k <= 1024, else DAWN_ERR_INVALID.
 * The rule: each list's first min(count, k) entries; an entry whose (distance, label) also occurs in a list
 * with a smaller index is dropped (a page stored on two shards); the rest ordered by (distance, label, list
 * index); the first k kept.  With every label stored once this is one index holding every list's rows; a
 * label stored on several shards at the same distance is returned as often as the lowest-index shard holding
 * it returns it.  Nothing past counts_out[b] is written. */
int dawn_merge_results_device(int device, const uint64_t *d_labels, const float *d_distances,
                              const uint32_t *d_counts, size_t n_lists, size_t list_stride_bytes,
                              size_t batch, size_t k, uint64_t *d_labels_out, float *d_distances_out,
                              uint32_t *d_counts_out, void *stream);
/* Fill rows [size, size+n) with the synthetic corpus (seed, first_row..) generated on the
 * device; labels are first_row + i + 1.  Test / bench aid: 100M vectors cannot cross PCIe in
 * a test budget.  Bit-identical to oracle/dawn_oracle.c:dawn_oracle_synth_rows_f16. */
int dawn_index_add_synthetic(dawn_index *idx, uint64_t seed, uint64_t first_row, size_t n);

/* ---- callers and formats either side of the path (SURVEY.md section 8f) ------------------------- */

/* Host mirrors of the reference's normalisation gate and helpers (src/search/vector.rs:181-197),
 * same sequential f32 arithmetic. */
float dawn_vector_length(const float *v384);
int dawn_is_normalized(const float *v384); /* 1 if finite and 0.99 < |v| < 1.01 */
void dawn_normalize(float *v384);
/* The i24 wire codec of query embeddings (src/search/vector.rs:48-87; UdpPacket::Search carries
 * 1152 bytes, src/net/udp_packets.rs:35-38).  decode returns DAWN_ERR_INVALID when the decoded
 * vector is not normalised, like the reference's ensure!(). */
void dawn_encode_i24(const float *v384, uint8_t *out1152);
int dawn_decode_i24(const uint8_t *in1152, float *out384);

/* distance_limit of UdpPacket::Search: hits with distance >= limit are not returned
 * (src/net/udp_service.rs:196-199).  NaN limit = no limit.  The limit is also pushed down into the
 * scan kernels as a score floor, so rows that cannot pass it are never kept, merged or re-scored. */
int dawn_index_search_limit(dawn_index *idx, const float *query384, size_t k, float distance_limit,
                            uint64_t *labels_out, float *distances_out, size_t *count_out);
/* The same for a batch (one limit for all queries): on the tensor-core path the limit becomes the initial
 * threshold of every query's candidate log. */
int dawn_index_search_batch_limit(dawn_index *idx, const float *queries, size_t batch, size_t k, float distance_limit,
                                  uint64_t *labels_out, float *distances_out, size_t *counts_out);
/* The peer side of a remote search: raw i24 query in (udp_service.rs:174-213). */
int dawn_index_search_i24(dawn_index *idx, const uint8_t *query1152, size_t k, int has_limit, float distance_limit,
                          uint64_t *labels_out, float *distances_out, size_t *count_out);
/* Stored vector in wire format (GetEmbedding over UDP, udp_service.rs:254-276). */
int dawn_index_get_i24(dawn_index *idx, uint64_t label, uint8_t *out1152);

/* Bulk load of a legacy `.emb` flat file: n repr(C) PageEntry records of 1568 bytes (url_pos u64,
 * title_pos u64, vector [f32;384], url_len u64, title_len u64; src/index/warc.rs:35-43), labels
 * first_label + i.  Records failing the normalisation gate are skipped and counted. */
int dawn_index_add_page_entries(dawn_index *idx, const void *entries, size_t n, uint64_t first_label,
                                size_t *skipped);

/* Micro-batching front.  The reference answers one query at a time from one thread
 * (src/search/search_service.rs:55-104); a batcher lets any number of threads call
 * dawn_batcher_search concurrently and answers them in batches of up to max_batch queries (one k
 * per batch).  A batch is what arrived while the previous one was on the GPU, plus the callers of
 * that previous batch if they come back within max_wait_us; a lone caller never waits.  Results
 * equal dawn_index_search's, bit for bit. */
typedef struct dawn_batcher dawn_batcher;
int dawn_batcher_create(dawn_index *idx, size_t max_batch, uint32_t max_wait_us, dawn_batcher **out);
/* The same front over a dawn_multi handle (below): single-query callers -> batches -> every shard -> merge. */
struct dawn_multi;
int dawn_batcher_create_multi(struct dawn_multi *m, size_t max_batch, uint32_t max_wait_us, dawn_batcher **out);
int dawn_batcher_search(dawn_batcher *b, const float *query384, size_t k, uint64_t *labels_out,
                        float *distances_out, size_t *count_out);
int dawn_batcher_stats(dawn_batcher *b, uint64_t *batches, uint64_t *queries, uint64_t *largest_batch);
const char *dawn_batcher_last_error(void);
void dawn_batcher_free(dawn_batcher *b);

/* ---- several GPUs, one process (the reference binary is one process, src/bin/dawnsearch.rs:59-128) ----
 * One handle owns one shard per listed device (NCCL communicators are created inside dawn_multi_create
 * with ncclCommInitAll).  add* places blocks of vectors round-robin on the shards; search* runs every
 * shard's exact top-k concurrently, exchanges the packed result blocks (k label/distance pairs per query)
 * with ONE ncclAllGather over NVLink / NVSwitch and merges them on the first device -- the role of
 * search_remote's scatter / gather / BestResults merge (src/search/search_service.rs:201-277).
 * Queries a shard cannot certify are re-run exactly on that shard before the exchange, so results are
 * bit-identical to a single index holding everything.  (The one-process-per-GPU variant under
 * torch.distributed is dawnsearch_b200/sharded.py.) */
typedef struct dawn_multi dawn_multi;
int dawn_multi_create(const int *devices, size_t n_devices, uint32_t scalar, dawn_multi **out);
void dawn_multi_free(dawn_multi *m);
int dawn_multi_reserve(dawn_multi *m, size_t n_total);
int dawn_multi_add(dawn_multi *m, uint64_t label, const float *vector384);
int dawn_multi_add_batch(dawn_multi *m, const uint64_t *labels, const float *vectors, size_t n);
int dawn_multi_add_synthetic(dawn_multi *m, uint64_t seed, uint64_t first_row, size_t n);
/* dawn_index_remove_batch on every shard (a label may be stored on any of them); *removed_out = the shards' counts summed.
 * If a shard fails, the error is returned and *removed_out still counts the rows the other shards removed. */
int dawn_multi_remove_batch(dawn_multi *m, const uint64_t *labels, size_t n, size_t *removed_out);
int dawn_multi_remove(dawn_multi *m, uint64_t label, size_t *removed_out);
int dawn_multi_search(dawn_multi *m, const float *query384, size_t k, uint64_t *labels_out, float *distances_out,
                      size_t *count_out);
int dawn_multi_search_batch(dawn_multi *m, const float *queries, size_t batch, size_t k, uint64_t *labels_out,
                            float *distances_out, size_t *counts_out);
/* distance_limit across the shards: every shard applies it before the exchange (NaN = none). */
int dawn_multi_search_limit(dawn_multi *m, const float *query384, size_t k, float distance_limit, uint64_t *labels_out,
                            float *distances_out, size_t *count_out);
int dawn_multi_search_batch_limit(dawn_multi *m, const float *queries, size_t batch, size_t k, float distance_limit,
                                  uint64_t *labels_out, float *distances_out, size_t *counts_out);
size_t dawn_multi_size(const dawn_multi *m);
size_t dawn_multi_capacity(const dawn_multi *m);
size_t dawn_multi_shards(const dawn_multi *m);
const char *dawn_multi_last_error(void);
/* "exchange": 0 = auto (NCCL all-gather; peer copies when a device is listed twice, there is one shard, or the result
 * blocks are under 16 KB -- a handful of queries, where one small peer copy per shard is quicker than a collective),
 * 1 = peer copies (cudaMemcpyPeerAsync into the first device), 2 = NCCL or fail.  Any other key is passed
 * to every shard's dawn_index_set_option. */
int dawn_multi_set_option(dawn_multi *m, const char *key, int64_t value);
typedef struct dawn_multi_stats {
    uint64_t searches, nccl_exchanges, peer_exchanges;
    uint64_t exact_reruns;     /* (shard, query) pairs re-run exactly because a certificate failed */
    uint64_t kernel_launches;  /* all shards */
    double last_search_ms;     /* CUDA-event time of the slowest shard's local search in the last call */
    double last_exchange_ms;   /* CUDA-event time of exchange + merge on the first device in the last call */
    uint32_t nccl_ready, reserved_;
} dawn_multi_stats;
int dawn_multi_get_stats(dawn_multi *m, dawn_multi_stats *out);
/* Persistence of the whole handle (DESIGN.md section 6).  dawn_multi_save writes ONE file, little-endian:
 *   0 "DAWNMULT", 8 u32 version = 1, 12 u32 scalar (DAWN_SCALAR_*), 16 u32 dims = 384, 20 u32 G (shards, 1..64),
 *   24 u64 add cursor (< G), 32 u64 rows[G], zeros up to byte 4096; then one section per shard, section 0 at 4096 and
 *   section g at the end of section g-1 rounded up to a multiple of 4096 (zero padding).  A section is u64 labels[rows],
 *   then the stored rows exactly as dawn_index_save writes them after its header.  The file ends with the last section.
 * Every shard writes its own section concurrently, to path.tmp, renamed when all are written; a failure removes the
 * temporary file and leaves path alone.  A save holds adds, removes, reserve, load and set_option off, never searches or
 * get.  Saving twice gives the same bytes, and so does save -> load (same shard count) -> save.
 * dawn_multi_load reads a DAWNMULT file or a dawn_index_save file (one section, cursor 0) into a handle with any number
 * of shards.  Same shard count: section g goes to shard g and the add cursor is restored.  Otherwise the N rows of all
 * sections, in order, are split as dawn_multi_add_synthetic splits: shard g gets rows [g P, min(N, (g+1) P)),
 * P = ceil(N / shards), cursor 0.  Stored rows are copied, never re-quantised.  Header, storage type, dimensions, shard
 * count, cursor, file length and rows per shard are checked first (DAWN_ERR_IO); the load fills every shard, then
 * publishes all of them at once, so a failure leaves the handle exactly as it was and no search sees a mix.  An empty
 * handle whose shards were reserved for their share is filled in place.  With every label stored once, answers do not
 * depend on placement; a label stored several times may come back differently after a load into another shard count,
 * as after any add (see dawn_merge_results_device). */
int dawn_multi_save(dawn_multi *m, const char *path);
int dawn_multi_load(dawn_multi *m, const char *path);
/* dawn_index_get on every shard: the lowest-index shard holding the label answers with its lowest row (the copy the merge
 * keeps).  DAWN_ERR_INVALID if no shard holds it; a CUDA error on any shard is returned as such. */
int dawn_multi_get(dawn_multi *m, uint64_t label, float *out384);
int dawn_multi_get_i24(dawn_multi *m, uint64_t label, uint8_t *out1152);
/* dawn_index_verify on every shard: bad_rows summed, min_norm over non-empty shards (0 if all are empty), max_norm the largest. */
int dawn_multi_verify(dawn_multi *m, size_t *bad_rows_out, float *min_norm_out, float *max_norm_out);
/* dawn_index_search_i24 over the handle: DAWN_ERR_INVALID when the decoded query is not normalised, else dawn_multi_search_limit. */
int dawn_multi_search_i24(dawn_multi *m, const uint8_t *query1152, size_t k, int has_limit, float distance_limit,
                          uint64_t *labels_out, float *distances_out, size_t *count_out);

/* ---- instrumentation ------------------------------------------------------------------- */
typedef struct dawn_profile {
    uint64_t scan_launches;  /* K2 launches since the last reset */
    double scan_ms;          /* summed CUDA-event time of those launches (on their stream) */
    uint64_t finalize_launches;
    double finalize_ms;
    uint64_t queries;        /* queries answered */
    uint64_t uncertified;    /* queries whose exactness certificate did not hold */
    uint64_t escalations;    /* queries re-run with a longer candidate list */
    uint64_t kernel_launches; /* all kernels launched by the library since the last reset */
    uint64_t gemm_batches;   /* batches answered by the tensor-core path (K3) */
    double gemm_ms;          /* summed CUDA-event time of those batches (all rounds, excl. finalize) */
    /* Counted ON THE DEVICE by every finalize launch, so they also cover dawn_index_search_device (which
     * cannot escalate: it only enqueues): results written without an exactness certificate, and the OR of
     * every scan status word (nonzero = internal buffer overflow, a bug). */
    uint64_t device_uncertified;
    uint64_t device_status;
    /* Largest |selection score - exact re-score| over every candidate any finalize launch has handled since the last reset
     * (all paths).  The certificate's eps constants must stay above it: tests/test_gpu_slack.py. */
    double max_selection_error;
    uint64_t shadow_batches; /* of gemm_batches: fp16 corpus answered through its int8 shadow (option "shadow_i8") */
} dawn_profile;
/* enable != 0: record CUDA events around every K2 / finalize launch (adds host syncs when
 * read).  Off by default. */
int dawn_index_set_profiling(dawn_index *idx, int enable);
/* Tuning knobs: "gemm_min_batch" (default 16) and "gemm_min_rows" (default 65536) decide when a
 * batch takes the tensor-core path instead of repeated streaming scans; "force_path" 0 = auto,
 * 1 = scan only, 2 = tensor-core path whenever the corpus holds >= 1024 vectors.
 * "gemm_small_batch" (2) / "gemm_small_batch_rows" (2M): on big corpora even small batches take the tensor-core path (fp16 and int8).
 * "shadow_i8" (0): 1 = an fp16 corpus also keeps an int8 copy of itself (+388 B per row, built lazily before a search) and
 * batches that would take the fp16 tensor-core path are FILTERED on the copy by the int8 tensor cores instead -- half the
 * HBM bytes, twice the MMA rate -- while every candidate is re-scored on the fp16 rows: results stay bit-identical.
 * "shadow_group_rows" (32; 1 or 32): rows of the copy that share one scale, in groups aligned to the row index.  32 makes the
 * filter's first level as tight as its per-element test; 1 = a scale per row.  A change drops the copy (it waits for searches
 * in flight) and the next search rebuilds it.  Results are the same either way.
 * "shadow_single_rows" (6M): with a shadow, from this many rows on even a single query takes that path (388 B per row
 * instead of the scan's 768 B).  "shadow_big_k_rows" (40M): batches of >= 128 queries with k > 32 take it only from this many
 * rows on (below, the exact re-scores of k + 4 candidates per round cost more than the int8 tiles save).
 * int8 corpora: "i8_tensor_min_batch" (16, 0 = never) -- from this batch size on the corpus is dequantised chunk by chunk
 * ("i8_tensor_chunk_rows", 4M) into an fp16 scratch and searched on the tensor cores; results stay bit-identical.
 * "gemm_cta_group", "gemm_chunk_tiles", "gemm_growth", "gemm_sequential_tiles": A/B knobs of the tensor-core path, 0 = automatic;
 * "gemm_unit_sync" (1): the CTA pairs that share a corpus chunk start it together (DRAM traffic 1.0x instead of up to 1.9x). */
int dawn_index_set_option(dawn_index *idx, const char *key, int64_t value);
int dawn_index_get_profile(dawn_index *idx, dawn_profile *out, int reset);

/* Evidence for the exactness certificate's constants (not a search path).  For `batch` host queries against an fp16 index of
 * at most 2048 rows, EVERY (query,row) score the tensor-core kernel produces is compared on the device with the f64 dot
 * product of the same fp16 operands, with the sequential f32 re-score and with the f64 dot product of the f32 query.
 * Maxima, pair count and a histogram of |tensor-core score - sequential score| accumulate in *acc across calls. */
typedef struct dawn_score_error {
    double max_mma_vs_f64;       /* |tcgen05 score - f64 dot(fp16(q), x)|: the MMA's own accumulation error */
    double max_seq_vs_f64;       /* |sequential f32 score - f64 dot(q, x)|: rounding of the exact re-score */
    double max_mma_vs_seq;       /* |tcgen05 score - sequential f32 score|: what eps_q has to bound */
    double max_err_over_eps_q;   /* max of that difference divided by the query's eps_q (must stay below 1) */
    uint64_t pairs;
    uint64_t hist[40];           /* hist[0]: difference == 0; hist[b]: difference in [2^(b-40), 2^(b-39)) */
    float scan_eps, gemm_accum_slack, i8_dequant_slack, reserved_;  /* the constants compiled into the library */
} dawn_score_error;
int dawn_debug_gemm_score_error(dawn_index *idx, const float *queries, size_t batch, dawn_score_error *acc);

#ifdef __cplusplus
}
#endif
#endif
