// dawn_common.cuh -- shared device/host definitions for libdawn_b200.so (sm_100a only).
//
// Domain vocabulary follows the reference (dawn-search/dawnsearch v0.2.0):
//   page vector / embedding : 384 x f32 unit vector     (src/search/vector.rs:26-28)
//   label                   : caller-supplied u64 page id (SQLite rowid,
//                             src/search/search_provider.rs:145,275)
//   distance                : 1 - dot, smaller is better  (src/search/vector.rs:128-134)
// "row" is the position of a page vector inside this GPU's corpus shard.
#pragma once

#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace dawn {

constexpr int kDim = 384;                       // EM_LEN, src/search/vector.rs:26
constexpr int kRowBytesF16 = kDim * 2;          // 768 B per stored fp16 page vector
constexpr int kMaxCand = 128;                   // largest candidate-list length (k + slack)
constexpr int kI8BlockRows = 8;                 // int8 storage: 8 rows of 384 int8, then their 8 f32 scales
constexpr int kI8BlockBytes = kI8BlockRows * kDim + kI8BlockRows * 4;  // 3,104 (a multiple of 16 for TMA)
constexpr uint32_t kNoRow = 0xFFFFFFFFu;
constexpr uint64_t kNoLabel = 0xFFFFFFFFFFFFFFFFull;

// One top-k candidate.  16 bytes so it moves as a single 128-bit access.
struct __align__(16) Cand {
    float score;     // dot product (approximate order of summation until re-scored)
    uint32_t row;    // row inside the shard, kNoRow for an empty slot
    uint64_t label;  // page id
};

__host__ __device__ inline Cand empty_cand() {
    Cand c;
#ifdef __CUDA_ARCH__
    c.score = __int_as_float(0xff800000);  // -inf
#else
    c.score = -__builtin_inff();
#endif
    c.row = kNoRow;
    c.label = kNoLabel;
    return c;
}

// Total order of the top-k: score descending, then label ascending (north_star:
// "deterministic tie-break on lower page id"), then row ascending so that the order is
// strict even if a caller adds the same label twice.  The reference's BestResults
// (src/search/best_results.rs:44-65) keeps whichever tied entry arrived first; ours is
// independent of arrival order.
__host__ __device__ inline bool cand_better(const Cand &a, const Cand &b) {
    if (a.score != b.score) return a.score > b.score;
    if (a.label != b.label) return a.label < b.label;
    return a.row < b.row;
}

// Monotone map float -> uint so that atomicMax on the uint orders like the float.
__device__ inline uint32_t float_to_ordered(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ inline float ordered_to_float(uint32_t u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}

// ---- synthetic corpus (test / bench aid).  Must stay bit-identical to
// oracle/dawn_oracle.c:dawn_oracle_synth_row_f32 -- integer hash, exact integer sum of
// squares, then correctly rounded IEEE f64 sqrt / divide / multiply only.
__host__ __device__ inline uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__host__ __device__ inline int32_t synth_raw(uint64_t seed, uint64_t row, uint32_t col) {
    uint64_t h = mix64(seed + 0x9E3779B97F4A7C15ull * (row * (uint64_t)kDim + col + 1));
    uint32_t s = (uint32_t)(h & 0xFFFF) + (uint32_t)((h >> 16) & 0xFFFF) +
                 (uint32_t)((h >> 32) & 0xFFFF) + (uint32_t)(h >> 48);
    return (int32_t)s - 131070;
}

// ---- kernel launchers (defined in the .cu files) -------------------------------------

// K1: f32 page vectors -> stored fp16 rows (round to nearest even), appended at dst.
// Replaces the per-vector work of usearch Index::add (src/search/search_provider.rs:149,284).
// saturate: clamp to +-65504 instead of rounding to inf (the selection copy of DAWN_SCALAR_F32 rows)
cudaError_t launch_ingest_f16(const float *src_f32, __half *dst, size_t n_rows, cudaStream_t s, bool saturate = false);
// Synthetic rows [first_row, first_row+n) written straight into the corpus arena.
cudaError_t launch_synth_f16(__half *dst, uint64_t seed, uint64_t first_row, size_t n_rows,
                             cudaStream_t s);
// the same rows before the fp16 rounding (DAWN_SCALAR_F32 storage); bit-identical to oracle/dawn_oracle.c:dawn_oracle_synth_row_f32
cudaError_t launch_synth_f32(float *dst, uint64_t seed, uint64_t first_row, size_t n_rows, cudaStream_t s);
// Gather stored rows back to f32 (dawn_index_get; SearchProvider::embedding_for_page,
// src/search/search_provider.rs:183-195, served from the device corpus).
cudaError_t launch_gather_f32(const __half *corpus, const uint32_t *rows, size_t n, float *out,
                              cudaStream_t s);
// labels[i] = first + i (synthetic corpora: label = row + 1, like SQLite rowids, search_provider.rs:275)
cudaError_t launch_iota_labels(uint64_t *dst, uint64_t first, size_t n, cudaStream_t s);
cudaError_t launch_shadow_quantize(const __half *corpus, uint8_t *arena, size_t first, size_t n, int group_rows,
                                   uint32_t *kappa_bits, cudaStream_t s);
cudaError_t launch_truncate_by_limit(const float *dist, uint32_t *counts, size_t batch, size_t k, float limit, cudaStream_t s);

struct ScanLaunch {
    const __half *corpus;     // [n_rows][384] fp16
    const uint64_t *labels;   // [n_rows]
    uint32_t n_rows;
    const float *queries;     // [nq][384] f32, device
    int nq;                   // queries in this pass (1, 2 or 4)
    int kprime;               // candidate list length: 16, 32, 64 or 128
    Cand *partials;           // [nq][grid][kprime] out
    uint32_t *chunk_counter;  // zeroed before launch
    uint32_t *status;         // device word, bit0 = internal buffer overflow (a bug if ever set)
    int grid;                 // number of CTAs (= SM count)
    float score_floor;        // rows scoring below this are never candidates (-inf = none); distance_limit pushed down
};
// K2: streaming scan + fused per-CTA top-k' (replaces usearch Index::search,
// src/search/search_provider.rs:214).
cudaError_t launch_scan_topk_f16(const ScanLaunch &p, cudaStream_t s);
int scan_max_queries_per_pass(int kprime);

struct FinalizeLaunch {
    const __half *corpus;
    const float *queries;   // [nq][384]
    int nq;
    const Cand *partials;   // [nq][n_lists][kprime], each list sorted by cand_better
    int n_lists;
    int kprime;
    int k;                  // results wanted per query (<= kprime)
    float eps;              // bound on |scan score - exact score| used by the certificate
    uint64_t *labels_out;   // [nq][k]
    float *distances_out;   // [nq][k]
    uint32_t *counts_out;   // [nq]
    uint32_t *flags_out;    // [nq] bit0 = exactness certified
    int scalar;             // 0 = fp16 rows (corpus is __half*), 1 = blocked int8 arena (corpus is uint8_t*),
                            // 2 = re-score from corpus32 (the f32 vectors as given); selection ran on the fp16 copies
    const float *corpus32;  // scalar == 2 only
    const float *eps_q;     // optional per-query eps (GEMM path: depends on the query's fp16 rounding)
    const uint32_t *overflow;  // optional per-query "candidate log overflowed" flags -> not certified
    uint32_t *counters;     // optional: [n_counters] words (status word first) that CTA 0 zeroes for the next search
    int n_counters;
    uint32_t *status_out;   // optional: receives counters[0] (scan status) before the reset
    float eps_scale;        // multiplies every eps: > 1 when stored rows are longer than the reference's norm gate allows
    uint32_t *stats;        // optional device words: [0] += queries left uncertified, [1] |= scan status,
                            // [2] = max over every finalized candidate of |selection score - exact score| (f32 bits)
};
// One thread per raw log entry of a debug_raw_scores run: accumulates max |gemm - f64 dot(q16,x)| (tensor-core accumulation),
// max |sequential f32 - f64 dot(q,x)| (the re-score's own rounding), max |gemm - sequential f32| / eps_q, a histogram of
// |gemm - sequential f32| by binary exponent, and the pair count.  out: 8 doubles-as-u64 maxima/ratios + 40 bins + count.
cudaError_t launch_score_error(const uint2 *log, const uint32_t *cnt, int n_queries, int log_cap, const __half *corpus,
                               const float *q32, const __half *q16, const float *eps_q, unsigned long long *out,
                               cudaStream_t s);
// K5+K6: merge per-CTA lists, re-score candidates in the reference's order of summation
// (src/search/vector.rs:128-134), final order and 1 - score.
cudaError_t launch_finalize(const FinalizeLaunch &p, cudaStream_t s);

// ---- int8 storage (K4) ----
// A query prepared for the int8 scan: q ~= s1*hi + s2*lo.
struct __align__(16) I8Query {
    int8_t hi[kDim];
    int8_t lo[kDim];
    float s1, s2;
    float pad_[2];
};
__host__ __device__ inline size_t i8_row_offset(size_t row) {
    return (row / kI8BlockRows) * (size_t)kI8BlockBytes + (row % kI8BlockRows) * (size_t)kDim;
}
__host__ __device__ inline size_t i8_scale_offset(size_t row) {
    return (row / kI8BlockRows) * (size_t)kI8BlockBytes + (size_t)kI8BlockRows * kDim + (row % kI8BlockRows) * 4;
}
__host__ __device__ inline size_t i8_arena_bytes(size_t rows) {
    return (rows + kI8BlockRows - 1) / kI8BlockRows * (size_t)kI8BlockBytes;
}
struct ScanLaunchI8 {
    const uint8_t *corpus;    // blocked int8 arena
    const uint64_t *labels;
    uint32_t n_rows;
    const I8Query *queries;   // [nq] prepared queries, device
    int nq;                   // 1 or 2
    int kprime;
    Cand *partials;           // [nq][grid][kprime]
    uint32_t *chunk_counter;
    uint32_t *status;
    int grid;
    const float *eps_q;       // [nq] bound on |scan score - exact score| per query (prep_queries_i8)
    float limit_score;        // 1 - distance_limit, -inf = none; the kernel's floor is limit_score - 2 eps_q
};
cudaError_t launch_scan_topk_i8(const ScanLaunchI8 &p, cudaStream_t s);
cudaError_t launch_prep_queries_i8(const float *q32, int n_queries, I8Query *out, float *eps_q, cudaStream_t s);
// f32 rows -> blocked int8 arena at rows [first_row, first_row+n) (per-row absmax/127 scale).
cudaError_t launch_ingest_i8(const float *src_f32, uint8_t *arena, size_t first_row, size_t n_rows, cudaStream_t s);
cudaError_t launch_synth_i8(uint8_t *arena, size_t dst_first_row, uint64_t seed, uint64_t first_row, size_t n_rows,
                            cudaStream_t s);
cudaError_t launch_gather_f32_i8(const uint8_t *arena, const uint32_t *rows, size_t n, float *out, cudaStream_t s);

// Large batches over an int8 corpus by way of the fp16 tensor-core tiles (i8_tensor.cu).
cudaError_t launch_dequant_i8_f16(const uint8_t *arena, size_t first_row, size_t n_rows, __half *out, cudaStream_t s);
cudaError_t launch_gather_chunk_lists(const Cand *chunk_lists, int n_queries, int kp, uint32_t row_offset, int chunk,
                                      int n_chunks, Cand *gathered, const uint32_t *overflow, uint32_t *overflow_any,
                                      cudaStream_t s);

struct GemmSearch {
    const __half *corpus;     // [n_rows][384] fp16
    const uint64_t *labels;   // [n_rows]
    uint64_t n_rows;
    const float *queries;     // [n_queries][384] f32, device
    int n_queries;
    int kprime;               // candidates kept per query (<= 128)
    int grid;                 // CTAs (= SM count)
    int cta_group;            // 0 = auto (pairs when more than 128 queries), 1 or 2 to force
    int chunk_tiles;          // 0 = auto; tiles per work unit (tuning override)
    int sequential_tiles;     // 1 = visit tiles in stored order instead of the strided permutation (A/B only)
    int growth;               // rows visited grow by this factor per round (0 = automatic: 8, or up to 32 for one query tile)
    int no_unit_sync;         // 1 = no rendezvous of the workers that share a corpus chunk (A/B only)
    void *workspace;          // gemm_workspace_bytes(n_queries)
    Cand *final_lists;        // out: [ceil128(n_queries)][kprime] sorted candidates (approximate scores)
    float accum_slack;        // bound on the tensor-core accumulation error added to every eps_q
    float limit_score;        // 1 - distance_limit (-inf = none): rows that cannot pass it never enter a candidate log
    const float **eps_out;    // out: device pointer to per-query eps
    const uint32_t **overflow_out;  // out: device pointer to per-query overflow flags
    int *launches_out;        // out: kernels launched
    // debug (dawn_debug_gemm_score_error): run ONE round over all tiles with thresholds at -inf, skip the select, and hand back
    // the raw logs -- every (query,row) score the tensor cores produced.  Needs n_rows <= 2048 (the log capacity).
    int debug_raw_scores;
    const uint2 **debug_log_out;     // [qp][2048] (score bits, row)
    const uint32_t **debug_cnt_out;  // [qp]
    const __half **debug_q16_out;    // [qp][384] the fp16-rounded queries the MMA used
};
// K3: tcgen05 GEMM + fused top-k' over geometrically growing rounds of rows (gemm_topk.cu).
cudaError_t launch_gemm_search(const GemmSearch &p, cudaStream_t s);
size_t gemm_workspace_bytes(int n_queries);


// K4c: tcgen05 kind::i8 GEMM + fused filter straight from the blocked int8 arena, exact re-score between rounds (gemm_i8.cu).
struct GemmSearchI8 {
    const uint8_t *arena;     // blocked int8 arena (8 rows + 8 f32 scales per 3104-byte block)
    const uint64_t *labels;   // [n_rows]
    uint64_t n_rows;
    const float *queries;     // [n_queries][384] f32, device
    int n_queries;
    int kprime;               // candidates kept per query (<= 128); exact scores, so k' >= k is all it takes
    int grid;                 // CTAs (= SM count)
    int cta_group;            // 0 = auto (pairs when more than 128 queries), 1 or 2 to force
    int chunk_tiles;          // 0 = auto
    int sequential_tiles;     // 1 = visit tiles in stored order (A/B only)
    int growth;               // 0 = automatic
    int no_unit_sync;         // 1 = no rendezvous of the workers that share a corpus chunk (A/B only)
    void *workspace;          // gemm_i8_workspace_bytes(n_queries)
    Cand *final_lists;        // out: [ceil256(n_queries)][kprime] candidates with EXACT scores (unsorted)
    float limit_score;        // 1 - distance_limit (-inf = none)
    float eps_scale;          // > 1 when stored rows are longer than the reference's norm gate allows
    const uint32_t **overflow_out;  // out: device pointer to per-query overflow flags
    int *launches_out;        // out: kernels launched
    // Shadow mode: `arena` is an int8 COPY of the fp16 rows at `rescore_f16` ([n_rows][384]), which hold the truth: the
    // rounds filter on the copy and re-score on the fp16 rows.  shadow_kappa bounds ||x16 - s_row x8|| / s_row over all rows.
    const __half *rescore_f16;
    float shadow_kappa;
};
cudaError_t launch_gemm_search_i8(const GemmSearchI8 &p, cudaStream_t s);
size_t gemm_i8_workspace_bytes(int n_queries);

// dawn_index_remove_batch (remove.cu).  mark: hash the m requested labels (d_req, device) and flag every row of
// labels[0, n) whose label is among them; meta_out (host) receives {r = rows flagged, h = flagged rows below n - r}.
// pair: holes[i] = i-th flagged row below n - r, donors[i] = i-th unflagged row in [n - r, n), i < h.  Both read the
// scratch of remove_scratch_bytes(m, n) that mark filled.
size_t remove_scratch_bytes(size_t m, size_t n);
cudaError_t launch_remove_mark(const uint64_t *d_req, size_t m, const uint64_t *labels, size_t n, void *scratch, uint32_t *meta_out,
                               cudaStream_t s);
cudaError_t launch_remove_pair(const void *scratch, size_t m, size_t n, uint32_t r, uint32_t h, uint32_t *holes, uint32_t *donors,
                               cudaStream_t s);
struct RemoveMove {
    const uint32_t *holes, *donors;
    size_t n_pairs;
    uint8_t *arena;     // fp16 rows, or the blocked int8 arena when i8
    int i8;
    float *corpus32;    // DAWN_SCALAR_F32 only, else null
    uint8_t *shadow;    // the int8 shadow of an fp16 corpus, or null
    uint64_t *labels;
};
// move: copy every row, scale and label of donors[i] into holes[i].
cudaError_t launch_remove_move(const RemoveMove &p, cudaStream_t s);

}  // namespace dawn
