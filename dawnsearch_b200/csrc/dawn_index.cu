// dawn_index.cu -- the C ABI (include/dawn_index.h) and the host-side index object:
// corpus arena in HBM, label table, pinned staging for adds, a pool of search workspaces, streams.
//
// This object takes the place of usearch's `Index` behind the reference's SearchProvider
// (/root/reference/src/search/search_provider.rs:67,102).  No CPU fallback exists: every
// compute path launches the kernels in scan_topk.cu / gemm_topk.cu / finalize.cu / ingest.cu.
//
// Concurrency model (SURVEY.md section 8b, "Threading"):
//   * `mu` guards the writer-side state: staged adds, size, capacity, reserve / load / save.
//   * `corpus_mu` (shared) guards the arena POINTERS.  A search holds it shared from its snapshot of
//     (pointers, size) until its results are on the host; only a reallocation (reserve growth, load)
//     takes it exclusively.  Appends write rows >= every snapshot, so they never wait for searches.
//   * Every host search leases its own SearchWs (stream + device / pinned buffers) from a pool, so
//     several host threads search one handle concurrently.  The device-resident entry point
//     (dawn_index_search_device) only enqueues; it uses one dedicated workspace chained by an event.
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <new>
#include <shared_mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/dawn_index.h"
#include "dawn_common.cuh"

using namespace dawn;

namespace {

thread_local std::string g_last_error;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

constexpr size_t kStageRowsHost = 8192;  // pinned staging: 8192 vectors = 12 MB of f32
// Bounds on |selection score - exact score| used by the exactness certificate.  They are DERIVED, not guessed:
// tests/test_gpu_slack.py measures the worst observed error of each selection kernel over >1e9 (query,row)
// pairs incl. adversarial same-sign rows (dawn_debug_score_error) and asserts every constant here exceeds the
// observed maximum at least twofold; the histogram is committed under profiles/.
constexpr float kScanEps = 3.0e-5f;         // K2: two f32 summation orders over 384 terms, |q||x| <= 1.03
constexpr float kGemmAccumSlack = 6.0e-5f;  // K3: tensor-core f32 accumulation over K=384 + the sequential re-score
constexpr float kF32StoreSlack = 5.1e-4f;   // DAWN_SCALAR_F32: selection runs on fp16 copies, |q.(fp16(x) - x)| <= 2^-11 |q||x| = 4.9e-4 * 1.01^2
constexpr float kRowNormGate = 1.0105f;     // the reference's gate (vector.rs:185-192) plus fp16 / int8 rounding
constexpr int kMaxPoolWs = 8;               // host searches in flight per handle
constexpr size_t kBulkMinRows = 32768;      // add_batch calls at least this large take the parallel bulk pipeline
constexpr int kBulkThreads = 12;       // copier threads (lanes) of the bulk-load pipeline; DAWN_BULK_THREADS uses fewer

// merge kernel for sharded searches, defined at the bottom of this file
cudaError_t launch_merge_results(const uint64_t *labels, const float *dist, const uint32_t *counts,
                                 int n_lists, size_t list_stride_bytes, int batch, int k, uint64_t *labels_out,
                                 float *dist_out, uint32_t *counts_out, cudaStream_t s);
cudaError_t launch_find_label(const uint64_t *labels, size_t n, uint64_t label, uint32_t *row_out,
                              cudaStream_t s);
// norm-gate scan over stored rows [first, first+n): stats[0] += rows outside (0.99,1.01) or non-finite,
// stats[1] = max(stats[1], bits of the largest finite norm), stats[2] = min(...) (as ordered uints)
cudaError_t launch_verify_rows(const void *arena, int scalar, size_t first, size_t n, uint32_t *stats, cudaStream_t s);

struct EventPair {
    cudaEvent_t a, b;
    int kind;  // 0 scan, 1 finalize, 2 gemm (all rounds of one batch)
};

// Everything ONE in-flight search needs.  Never shared between two searches at a time.
struct SearchWs {
    cudaStream_t stream = nullptr;  // owned
    size_t n_rows = 0;              // snapshot of the index size this search sees
    float eps_scale = 1.0f;         // > 1 when stored rows exceed the reference's norm gate
    bool odd_rows = false;          // some stored row has an inf / NaN / fp16-overflowing component: only the scan is exact
    size_t q_cap = 0;               // queries
    float *d_queries = nullptr, *h_queries = nullptr;
    // results of the host API: ONE packed block (labels | distances | counts | flags | status) so that a
    // search costs a single D2H copy
    uint8_t *d_result = nullptr, *h_result = nullptr;
    size_t result_cap = 0;
    float limit_score = -INFINITY;  // 1 - distance_limit of the search being enqueued (pushed down into the kernels)
    bool counters_clean = false;    // finalize leaves the chunk counters / status word zeroed for the next search
    Cand *d_partials = nullptr;
    size_t partials_cap = 0;
    uint32_t *d_counters = nullptr;  // one chunk counter per scan pass, + status word at [0]
    size_t counters_cap = 0;
    void *d_gemm_ws = nullptr;  // K3 workspace (fp16 queries, eps, thresholds, candidate logs)
    size_t gemm_ws_cap = 0;
    __half *d_i8_scratch = nullptr;  // one dequantised chunk (fp16-tile int8 path)
    size_t i8_scratch_rows = 0;
    Cand *d_i8_lists = nullptr;  // [batch][n_chunks][k'] gathered candidate lists
    size_t i8_lists_cap = 0;
    uint32_t *d_i8_overflow = nullptr;  // [batch] log overflow in any chunk
    size_t i8_overflow_cap = 0;
    // device API only: searches enqueued on different caller streams are chained by this event
    cudaEvent_t ws_done = nullptr;
    cudaStream_t ws_stream = nullptr;
    bool ws_used = false;
    // instrumentation, merged into the index when the lease ends
    std::vector<EventPair> pending, free_events;
    dawn_profile prof{};
};

struct BulkLane {  // one copier thread of the bulk-load pipeline
    cudaStream_t stream = nullptr;
    float *h_buf[2] = {nullptr, nullptr};
    uint64_t *h_lab[2] = {nullptr, nullptr};
    float *d_buf[2] = {nullptr, nullptr};
    cudaEvent_t done[2] = {nullptr, nullptr};
    bool busy[2] = {false, false};
};

}  // namespace

struct dawn_index {
    std::mutex mu;                 // writer-side state (see the header comment)
    std::shared_mutex corpus_mu;   // arena pointers
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;  // ingest / maintenance stream
    std::atomic<bool> dead{false};  // sticky CUDA failure

    int scalar = DAWN_SCALAR_F16;  // storage of the corpus: fp16 rows or the blocked int8 arena
    __half *corpus = nullptr;      // fp16: [phys][384]; int8: the same pointer holds the blocked arena
    float *corpus32 = nullptr;     // DAWN_SCALAR_F32 only: the vectors as given, [phys][384] f32 (what the exact re-score reads)
    uint64_t *labels = nullptr;
    // int8 shadow of an fp16 corpus (option "shadow_i8"): a quantised COPY in the blocked int8 layout, used only to FILTER on
    // the int8 tensor cores / at half the HBM bytes; candidates are re-scored on the fp16 rows, so answers do not change.
    // Built lazily before a search (rows [shadow_rows, size)), dropped whenever the arena is replaced.
    std::atomic<uint8_t *> shadow{nullptr};
    std::atomic<size_t> shadow_rows{0};
    std::atomic<float> shadow_kappa{0.f};  // max over shadow rows of ||x16 - s_row x8|| / s_row, measured by the quantiser
    uint32_t *d_shadow_kappa = nullptr;    // device scalar (f32 bits, atomicMax)
    std::atomic<size_t> size{0};      // rows committed to the device
    std::atomic<size_t> capacity{0};  // logical capacity promised to the caller
    size_t phys = 0;                  // rows actually allocated

    // staged adds (host, pinned) not yet on the device
    // Two buffers: while the GPU copies / converts one, the host fills the other.
    float *h_stage_buf[2] = {nullptr, nullptr};
    uint64_t *h_labels_buf[2] = {nullptr, nullptr};
    float *d_stage_buf[2] = {nullptr, nullptr};
    cudaEvent_t stage_done[2] = {nullptr, nullptr};
    bool stage_busy[2] = {false, false};
    int stage_cur = 0;
    float *h_stage = nullptr;
    uint64_t *h_stage_labels = nullptr;
    std::atomic<size_t> staged{0};
    float *d_stage = nullptr;
    BulkLane bulk[kBulkThreads];
    bool bulk_ready = false;

    // norm bookkeeping for the certificate: rows [0, norm_checked) have been through the gate scan
    uint32_t *d_norm_stats = nullptr;  // [0] bad rows, [1] max norm (ordered bits), [2] min norm, [3] odd rows (verify_rows_kernel)
    uint32_t *h_norm_stats = nullptr;  // pinned
    size_t norm_checked = 0;
    uint64_t bad_rows = 0, odd_rows = 0;
    float norm_max = 0.f, norm_min = INFINITY;

    // device-side counters: [0] queries returned without a certificate by any finalize launch,
    // [1] OR of every scan status word (internal buffer overflow; a bug if ever nonzero)
    uint32_t *d_stats = nullptr;
    uint32_t *h_stats = nullptr;  // pinned

    // path selection: batches >= gemm_min_batch over >= gemm_min_rows rows take the tensor-core path
    std::atomic<int64_t> gemm_min_batch{16};
    std::atomic<int64_t> gemm_min_rows{65536};
    std::atomic<int64_t> gemm_small_batch{2};  // from this batch size on, big corpora also take the tensor path (r02 C4 sweeps: batch 2
                                               // costs 6.35 ms as a QT=2 scan and 5.7 ms on the tensor path at 50M rows)
    std::atomic<int64_t> gemm_small_batch_rows{2000000};
    std::atomic<int64_t> force_path{0};  // 0 auto, 1 scan only, 2 gemm whenever possible
    std::atomic<int64_t> gemm_cta_group{0};  // 0 auto, 1 = one CTA per tile, 2 = CTA pairs
    std::atomic<int64_t> gemm_chunk_tiles{0};
    std::atomic<int64_t> gemm_sequential_tiles{0};
    std::atomic<int64_t> gemm_growth{0};
    std::atomic<int64_t> gemm_unit_sync{1};  // rendezvous of the workers sharing a corpus chunk (gemm_pipe.cuh)
    // int8 corpora: batches of at least this many queries take the tensor cores.  0 = never.
    std::atomic<int64_t> i8_tensor_min_batch{16};
    std::atomic<int64_t> i8_tensor_chunk_rows{4 << 20};
    std::atomic<int64_t> shadow_i8{0};  // 1 = keep an int8 shadow of an fp16 corpus (+388 B per row) and filter on it
    std::atomic<int64_t> shadow_group_rows{32};  // rows sharing one scale in the shadow (1 or 32, shadow_quantize_kernel)
    std::atomic<int64_t> shadow_big_k_rows{40000000};  // compute-bound batches with k > 32 take the shadow only from this many rows on
    std::atomic<int64_t> shadow_single_rows{6000000};  // with a shadow: from this many rows on, single queries take it too
    std::atomic<int64_t> i8_native{1};  // 1 = tcgen05 kind::i8 straight from the int8 arena, 0 = dequantise to fp16 tiles

    // search workspaces
    std::mutex pool_mu;
    std::condition_variable pool_cv;
    std::vector<SearchWs *> pool_free;
    int pool_total = 0;
    std::mutex dev_mu;  // serialises the enqueue of device-API searches
    SearchWs *dev_ws = nullptr;

    std::atomic<bool> profiling{false};
    std::mutex prof_mu;
    dawn_profile prof{};
};

namespace {

#define CK(idx, expr)                                                                         \
    do {                                                                                      \
        cudaError_t e__ = (expr);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            (idx)->dead = true;                                                               \
            return fail(DAWN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                  \
        }                                                                                     \
    } while (0)

int check_alive(dawn_index *idx) {
    if (!idx) return fail(DAWN_ERR_INVALID, "null index handle");
    if (idx->dead) return fail(DAWN_ERR_CUDA, "index is in a failed state after an earlier CUDA error");
    cudaError_t e = cudaSetDevice(idx->device);
    if (e != cudaSuccess) {
        idx->dead = true;
        return fail(DAWN_ERR_CUDA, "cudaSetDevice(%d): %s", idx->device, cudaGetErrorString(e));
    }
    return DAWN_OK;
}

// ---- workspaces ------------------------------------------------------------------------------

void free_ws(SearchWs *ws) {
    if (!ws) return;
    if (ws->stream) cudaStreamSynchronize(ws->stream);
    for (auto &p : ws->pending) ws->free_events.push_back(p);
    for (auto &p : ws->free_events) {
        cudaEventDestroy(p.a);
        cudaEventDestroy(p.b);
    }
    cudaFree(ws->d_queries);
    cudaFreeHost(ws->h_queries);
    cudaFree(ws->d_result);
    cudaFreeHost(ws->h_result);
    cudaFree(ws->d_i8_scratch);
    cudaFree(ws->d_i8_lists);
    cudaFree(ws->d_i8_overflow);
    cudaFree(ws->d_partials);
    cudaFree(ws->d_counters);
    cudaFree(ws->d_gemm_ws);
    if (ws->ws_done) cudaEventDestroy(ws->ws_done);
    if (ws->stream) cudaStreamDestroy(ws->stream);
    delete ws;
}

SearchWs *new_ws() {
    SearchWs *ws = new (std::nothrow) SearchWs();
    if (!ws) return nullptr;
    if (cudaStreamCreateWithFlags(&ws->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ws->ws_done, cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        free_ws(ws);
        return nullptr;
    }
    return ws;
}

void drain_events(SearchWs *ws, cudaStream_t s) {
    if (ws->pending.empty()) return;
    cudaStreamSynchronize(s);
    for (auto &p : ws->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            if (p.kind == 0) ws->prof.scan_ms += ms;
            else if (p.kind == 1) ws->prof.finalize_ms += ms;
            else ws->prof.gemm_ms += ms;
        }
        ws->free_events.push_back(p);
    }
    ws->pending.clear();
}

void merge_profile(dawn_index *idx, SearchWs *ws) {
    std::lock_guard<std::mutex> lk(idx->prof_mu);
    dawn_profile &d = idx->prof, &s = ws->prof;
    d.scan_launches += s.scan_launches;
    d.scan_ms += s.scan_ms;
    d.finalize_launches += s.finalize_launches;
    d.finalize_ms += s.finalize_ms;
    d.queries += s.queries;
    d.uncertified += s.uncertified;
    d.escalations += s.escalations;
    d.kernel_launches += s.kernel_launches;
    d.gemm_batches += s.gemm_batches;
    d.gemm_ms += s.gemm_ms;
    d.shadow_batches += s.shadow_batches;
    s = dawn_profile{};
}

// RAII lease of a pooled workspace for one host call.
struct WsLease {
    dawn_index *idx;
    SearchWs *ws = nullptr;
    explicit WsLease(dawn_index *i) : idx(i) {
        std::unique_lock<std::mutex> lk(idx->pool_mu);
        while (idx->pool_free.empty() && idx->pool_total >= kMaxPoolWs) idx->pool_cv.wait(lk);
        if (!idx->pool_free.empty()) {
            ws = idx->pool_free.back();
            idx->pool_free.pop_back();
            return;
        }
        idx->pool_total++;
        lk.unlock();
        ws = new_ws();
        if (!ws) {
            lk.lock();
            idx->pool_total--;
        }
    }
    ~WsLease() {
        if (!ws) return;
        drain_events(ws, ws->stream);
        merge_profile(idx, ws);
        ws->limit_score = -INFINITY;
        {
            std::lock_guard<std::mutex> lk(idx->pool_mu);
            idx->pool_free.push_back(ws);
        }
        idx->pool_cv.notify_one();
    }
};

bool begin_event(dawn_index *idx, SearchWs *ws, int kind, cudaStream_t s, EventPair *out) {
    if (!idx->profiling) return false;
    EventPair p;
    if (!ws->free_events.empty()) {
        p = ws->free_events.back();
        ws->free_events.pop_back();
    } else {
        if (cudaEventCreate(&p.a) != cudaSuccess || cudaEventCreate(&p.b) != cudaSuccess) return false;
    }
    p.kind = kind;
    cudaEventRecord(p.a, s);
    *out = p;
    return true;
}

void end_event(SearchWs *ws, EventPair &p, cudaStream_t s) {
    cudaEventRecord(p.b, s);
    ws->pending.push_back(p);
}

// ---- arena ------------------------------------------------------------------------------------

inline size_t arena_bytes(const dawn_index *idx, size_t rows) {
    return idx->scalar == DAWN_SCALAR_I8 ? i8_arena_bytes(rows) : rows * (size_t)kRowBytesF16;
}
inline uint8_t *arena_i8(const dawn_index *idx) { return reinterpret_cast<uint8_t *>(idx->corpus); }

// A device-API search may still be reading the arena on its caller's stream.
void wait_device_searches(dawn_index *idx) {
    if (idx->dev_ws && idx->dev_ws->ws_used) cudaEventSynchronize(idx->dev_ws->ws_done);
}

void drop_shadow(dawn_index *idx);

int alloc_arena(dawn_index *idx, size_t rows, __half **corpus_out, uint64_t **labels_out, float **corpus32_out) {
    __half *nc = nullptr;
    uint64_t *nl = nullptr;
    *corpus32_out = nullptr;
    if (idx->scalar == DAWN_SCALAR_F32) {
        cudaError_t e32 = cudaMalloc(corpus32_out, rows * (size_t)kDim * sizeof(float));
        if (e32 != cudaSuccess) {
            cudaGetLastError();
            *corpus32_out = nullptr;
            return fail(DAWN_ERR_CAPACITY, "cannot allocate %zu bytes of HBM for %zu f32 vectors: %s", rows * (size_t)kDim * 4, rows,
                        cudaGetErrorString(e32));
        }
    }
    cudaError_t e = cudaMalloc(&nc, arena_bytes(idx, rows));
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaFree(*corpus32_out);
        *corpus32_out = nullptr;
        return fail(DAWN_ERR_CAPACITY, "cannot allocate %zu bytes of HBM for %zu vectors: %s", arena_bytes(idx, rows), rows,
                    cudaGetErrorString(e));
    }
    e = cudaMalloc(&nl, rows * sizeof(uint64_t));
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaFree(nc);
        cudaFree(*corpus32_out);
        *corpus32_out = nullptr;
        return fail(DAWN_ERR_CAPACITY, "cannot allocate label table for %zu vectors", rows);
    }
    *corpus_out = nc;
    *labels_out = nl;
    return DAWN_OK;
}

// Called with idx->mu held.  Growth copies into a fresh arena and swaps the pointers under the
// exclusive corpus lock, i.e. after every in-flight search has finished with the old one.
int grow_physical(dawn_index *idx, size_t rows) {
    if (rows <= idx->phys) return DAWN_OK;
    if (rows > 0xFFFFFFF0ull) return fail(DAWN_ERR_INVALID, "capacity %zu exceeds 2^32 rows per GPU", rows);
    size_t want = rows;
    if (idx->phys > 0) {  // amortise the reference's reserve(size + 1024) pattern
        size_t geo = idx->phys + idx->phys / 2;
        if (geo > want) want = geo;
    }
    __half *nc = nullptr;
    uint64_t *nl = nullptr;
    float *n32 = nullptr;
    int rc = alloc_arena(idx, want, &nc, &nl, &n32);
    if (rc != DAWN_OK && want > rows) {
        want = rows;
        rc = alloc_arena(idx, want, &nc, &nl, &n32);
    }
    if (rc != DAWN_OK) return rc;
    const size_t n = idx->size;
    if (n > 0) {
        if (n32) CK(idx, cudaMemcpyAsync(n32, idx->corpus32, n * (size_t)kDim * sizeof(float), cudaMemcpyDeviceToDevice, idx->stream));
        CK(idx, cudaMemcpyAsync(nc, idx->corpus, arena_bytes(idx, n), cudaMemcpyDeviceToDevice, idx->stream));
        CK(idx, cudaMemcpyAsync(nl, idx->labels, n * sizeof(uint64_t), cudaMemcpyDeviceToDevice, idx->stream));
        CK(idx, cudaStreamSynchronize(idx->stream));
    }
    __half *oc;
    uint64_t *ol;
    float *o32;
    {
        std::unique_lock<std::shared_mutex> wr(idx->corpus_mu);
        wait_device_searches(idx);
        oc = idx->corpus;
        ol = idx->labels;
        o32 = idx->corpus32;
        idx->corpus = nc;
        idx->labels = nl;
        idx->corpus32 = n32;
        idx->phys = want;
        drop_shadow(idx);
    }
    if (oc) cudaFree(oc);
    if (ol) cudaFree(ol);
    if (o32) cudaFree(o32);
    return DAWN_OK;
}

// Enqueue the current staging buffer (H2D of the f32 rows, K1 convert, labels) WITHOUT waiting, and
// switch to the other buffer (waiting only if that one is still in flight).  idx->mu held.
int flush_staged_async(dawn_index *idx) {
    if (idx->staged == 0) return DAWN_OK;
    const size_t n = idx->staged;
    const size_t at = idx->size;
    const int cur = idx->stage_cur;
    CK(idx, cudaMemcpyAsync(idx->d_stage, idx->h_stage, n * kDim * sizeof(float), cudaMemcpyHostToDevice, idx->stream));
    if (idx->scalar == DAWN_SCALAR_I8) CK(idx, launch_ingest_i8(idx->d_stage, arena_i8(idx), at, n, idx->stream));
    else CK(idx, launch_ingest_f16(idx->d_stage, idx->corpus + at * kDim, n, idx->stream, idx->corpus32 != nullptr));
    if (idx->corpus32)  // the vectors as given, for the exact f32 re-score
        CK(idx, cudaMemcpyAsync(idx->corpus32 + at * kDim, idx->d_stage, n * kDim * sizeof(float), cudaMemcpyDeviceToDevice, idx->stream));
    CK(idx, cudaMemcpyAsync(idx->labels + at, idx->h_stage_labels, n * sizeof(uint64_t), cudaMemcpyHostToDevice, idx->stream));
    CK(idx, cudaEventRecord(idx->stage_done[cur], idx->stream));
    idx->stage_busy[cur] = true;
    idx->size = at + n;  // searches flush + synchronise before they snapshot the size
    idx->staged = 0;
    {
        std::lock_guard<std::mutex> lk(idx->prof_mu);
        idx->prof.kernel_launches++;
    }
    const int nxt = cur ^ 1;
    if (idx->stage_busy[nxt]) {
        CK(idx, cudaEventSynchronize(idx->stage_done[nxt]));
        idx->stage_busy[nxt] = false;
    }
    idx->stage_cur = nxt;
    idx->h_stage = idx->h_stage_buf[nxt];
    idx->h_stage_labels = idx->h_labels_buf[nxt];
    idx->d_stage = idx->d_stage_buf[nxt];
    return DAWN_OK;
}

// Make every staged / in-flight add visible: flush what is staged and wait for the stream.  idx->mu held.
int flush_staged(dawn_index *idx) {
    if (idx->staged == 0 && !idx->stage_busy[0] && !idx->stage_busy[1]) return DAWN_OK;
    int rc = flush_staged_async(idx);
    if (rc) return rc;
    CK(idx, cudaStreamSynchronize(idx->stream));
    idx->stage_busy[0] = idx->stage_busy[1] = false;
    return DAWN_OK;
}

// The certificate's eps constants assume stored rows inside the reference's norm gate.  Rows added since the
// last search go through the gate scan once (HBM-bound, 768 B / 388 B per row); if any stored row is longer
// than the gate allows every eps is scaled by the excess, so the certificate stays rigorous for callers that
// skip the gate (the raw ABI accepts any vector, like usearch does).  idx->mu held, stream idle.
int ensure_norms_checked(dawn_index *idx) {
    const size_t n = idx->size;
    if (idx->norm_checked >= n) return DAWN_OK;
    CK(idx, launch_verify_rows(idx->corpus, idx->scalar == DAWN_SCALAR_I8 ? 1 : 0, idx->norm_checked, n - idx->norm_checked, idx->d_norm_stats, idx->stream));
    CK(idx, cudaMemcpyAsync(idx->h_norm_stats, idx->d_norm_stats, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, idx->stream));
    CK(idx, cudaStreamSynchronize(idx->stream));
    idx->bad_rows = idx->h_norm_stats[0];
    idx->odd_rows = idx->h_norm_stats[3];
    memcpy(&idx->norm_max, &idx->h_norm_stats[1], 4);
    uint32_t inv = ~idx->h_norm_stats[2];
    memcpy(&idx->norm_min, &inv, 4);
    idx->norm_checked = n;
    return DAWN_OK;
}

// DAWN_SCALAR_F32 selects on fp16 copies saturated at +-65504: a copy that saturated (or holds inf / NaN) is off by more than
// any slack, so such an index answers but certifies nothing.
inline float eps_scale_of(const dawn_index *idx) {
    if (idx->odd_rows && idx->scalar == DAWN_SCALAR_F32) return INFINITY;
    return idx->norm_max > kRowNormGate ? idx->norm_max / 1.01f * 1.001f : 1.0f;
}

void reset_norm_stats(dawn_index *idx) {
    const uint32_t init[4] = {0u, 0u, 0u, 0u};  // max starts at +0.0; min is stored inverted (~bits), so 0 = +inf-ish
    cudaMemcpyAsync(idx->d_norm_stats, init, sizeof init, cudaMemcpyHostToDevice, idx->stream);
    cudaStreamSynchronize(idx->stream);
    idx->norm_checked = 0;
    idx->bad_rows = 0;
    idx->odd_rows = 0;
    idx->norm_max = 0.f;
    idx->norm_min = INFINITY;
}

// The arena was replaced (exclusive corpus lock held, no search in flight): the shadow goes with it.
void drop_shadow(dawn_index *idx) {
    uint8_t *p = idx->shadow.exchange(nullptr);
    if (p) cudaFree(p);
    idx->shadow_rows = 0;
    idx->shadow_kappa = 0.f;
}

// Bring the int8 shadow up to date with the fp16 corpus before a search (idx->mu held, stream idle).  Rows are only ever
// appended, so searches in flight -- which read rows below their own snapshot -- are not disturbed.  A failed allocation
// switches the option off: the fp16 path answers instead.
int ensure_shadow(dawn_index *idx) {
    if (!idx->shadow_i8 || idx->scalar != DAWN_SCALAR_F16) return DAWN_OK;
    const size_t n = idx->size;
    if (n < 65536 || idx->shadow_rows >= n) return DAWN_OK;
    if (!idx->shadow) {
        const size_t bytes = (idx->phys + kI8BlockRows - 1) / kI8BlockRows * (size_t)kI8BlockBytes;
        uint8_t *p = nullptr;
        if (cudaMalloc(&p, bytes) != cudaSuccess || (!idx->d_shadow_kappa && cudaMalloc(&idx->d_shadow_kappa, 4) != cudaSuccess)) {
            cudaGetLastError();
            if (p) cudaFree(p);
            idx->shadow_i8 = 0;
            return DAWN_OK;
        }
        CK(idx, cudaMemsetAsync(p, 0, bytes, idx->stream));
        CK(idx, cudaMemsetAsync(idx->d_shadow_kappa, 0, 4, idx->stream));
        idx->shadow = p;
        idx->shadow_rows = 0;
        idx->shadow_kappa = 0.f;
    }
    const size_t first = idx->shadow_rows;
    CK(idx, launch_shadow_quantize(idx->corpus, idx->shadow, first, n - first, (int)idx->shadow_group_rows, idx->d_shadow_kappa,
                                   idx->stream));
    uint32_t bits = 0;
    CK(idx, cudaMemcpyAsync(&bits, idx->d_shadow_kappa, 4, cudaMemcpyDeviceToHost, idx->stream));
    CK(idx, cudaStreamSynchronize(idx->stream));
    float kappa;
    memcpy(&kappa, &bits, 4);
    idx->shadow_kappa = kappa * 1.0001f + 1e-4f;
    idx->shadow_rows = n;
    return DAWN_OK;
}

// DAWN_DEBUG_STAGES=1: wait for each kernel of a search separately (polling, 5 s) and say on stderr which one
// did not finish.  Debug aid only; never set in tests or benches.
bool debug_stages() {
    static const bool on = getenv("DAWN_DEBUG_STAGES") != nullptr;
    return on;
}
void debug_wait(SearchWs *ws, cudaStream_t s, const char *stage) {
    if (!debug_stages()) return;
    const auto t0 = std::chrono::steady_clock::now();
    while (true) {
        cudaError_t e = cudaStreamQuery(s);
        if (e == cudaSuccess) {
            fprintf(stderr, "[dawn debug] %s done\n", stage);
            return;
        }
        if (e != cudaErrorNotReady) {
            fprintf(stderr, "[dawn debug] %s: %s\n", stage, cudaGetErrorString(e));
            return;
        }
        if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 5.0) {
            uint32_t c[4] = {0, 0, 0, 0};
            cudaStream_t side;
            cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking);
            if (ws->d_counters) {
                cudaMemcpyAsync(c, ws->d_counters, sizeof(c), cudaMemcpyDeviceToHost, side);
                cudaStreamSynchronize(side);
            }
            fprintf(stderr, "[dawn debug] %s STILL RUNNING after 5 s (rows %zu, counters %u %u %u %u)\n", stage, ws->n_rows, c[0],
                    c[1], c[2], c[3]);
            fflush(stderr);
            return;
        }
    }
}

int choose_kprime(size_t k) {
    size_t want = k + (k / 8 > 4 ? k / 8 : 4);
    int kp = 16;
    while ((size_t)kp < want) kp <<= 1;
    return kp > kMaxCand ? kMaxCand : kp;
}

struct ResultView {
    uint64_t *labels;
    float *dist;
    uint32_t *counts, *flags, *status;
    size_t bytes;
};
constexpr size_t kDirectResultBytes = 4096;  // result blocks up to this size are written to host memory by the kernel

inline ResultView result_view(uint8_t *base, size_t batch, size_t k) {
    ResultView v;
    v.labels = reinterpret_cast<uint64_t *>(base);
    v.dist = reinterpret_cast<float *>(base + batch * k * 8);
    v.counts = reinterpret_cast<uint32_t *>(base + batch * k * 12);
    v.flags = v.counts + batch;
    v.status = v.flags + batch;
    v.bytes = batch * k * 12 + batch * 8 + 16;
    return v;
}

int ensure_query_ws(dawn_index *idx, SearchWs *ws, size_t batch, size_t k) {
    if (batch > ws->q_cap) {
        size_t cap = batch < 64 ? 64 : batch;
        if (ws->d_queries) cudaFree(ws->d_queries);
        if (ws->h_queries) cudaFreeHost(ws->h_queries);
        ws->d_queries = nullptr;
        ws->h_queries = nullptr;
        ws->q_cap = 0;
        CK(idx, cudaMalloc(&ws->d_queries, cap * kDim * sizeof(float)));
        CK(idx, cudaMallocHost(&ws->h_queries, cap * kDim * sizeof(float)));
        ws->q_cap = cap;
    }
    const size_t need = batch * (k ? k : 1) * 12 + batch * 8 + 16;
    if (need > ws->result_cap) {
        size_t cap = need < 65536 ? 65536 : need;
        if (ws->d_result) cudaFree(ws->d_result);
        if (ws->h_result) cudaFreeHost(ws->h_result);
        ws->d_result = nullptr;
        ws->h_result = nullptr;
        ws->result_cap = 0;
        CK(idx, cudaMalloc(&ws->d_result, cap));
        CK(idx, cudaMallocHost(&ws->h_result, cap));
        ws->result_cap = cap;
    }
    return DAWN_OK;
}

template <typename T>
int ensure_dev(dawn_index *idx, T **ptr, size_t *cap, size_t need_elems) {
    if (need_elems <= *cap) return DAWN_OK;
    if (*ptr) cudaFree(*ptr);
    *ptr = nullptr;
    *cap = 0;
    CK(idx, cudaMalloc(ptr, need_elems * sizeof(T)));
    *cap = need_elems;
    return DAWN_OK;
}
int ensure_gemm_ws(dawn_index *idx, SearchWs *ws, size_t bytes) {
    if (bytes <= ws->gemm_ws_cap) return DAWN_OK;
    if (ws->d_gemm_ws) cudaFree(ws->d_gemm_ws);
    ws->d_gemm_ws = nullptr;
    ws->gemm_ws_cap = 0;
    CK(idx, cudaMalloc(&ws->d_gemm_ws, bytes));
    ws->gemm_ws_cap = bytes;
    return DAWN_OK;
}

// Zero the chunk counters / status word unless the previous search's finalize already did.
int prepare_counters(dawn_index *idx, SearchWs *ws, size_t need, cudaStream_t s) {
    if (need > ws->counters_cap) {
        size_t cap = need < 1024 ? 1024 : need;
        if (ws->d_counters) cudaFree(ws->d_counters);
        ws->d_counters = nullptr;
        ws->counters_cap = 0;
        CK(idx, cudaMalloc(&ws->d_counters, cap * sizeof(uint32_t)));
        ws->counters_cap = cap;
        ws->counters_clean = false;
    }
    if (!ws->counters_clean) CK(idx, cudaMemsetAsync(ws->d_counters, 0, ws->counters_cap * sizeof(uint32_t), s));
    ws->counters_clean = false;  // dirty until this search's finalize has been enqueued
    return DAWN_OK;
}

void fill_gemm_knobs(const dawn_index *idx, GemmSearch &gs) {
    gs.grid = idx->sm_count;
    gs.cta_group = (int)idx->gemm_cta_group;
    gs.chunk_tiles = (int)idx->gemm_chunk_tiles;
    gs.sequential_tiles = (int)idx->gemm_sequential_tiles;
    gs.growth = (int)idx->gemm_growth;
    gs.no_unit_sync = idx->gemm_unit_sync ? 0 : 1;
}

int run_finalize(dawn_index *idx, SearchWs *ws, FinalizeLaunch &fl, cudaStream_t s, size_t batch) {
    fl.eps_scale = ws->eps_scale;
    fl.stats = idx->d_stats;
    EventPair evf;
    bool timedf = begin_event(idx, ws, 1, s, &evf);
    CK(idx, launch_finalize(fl, s));
    if (timedf) end_event(ws, evf, s);
    ws->prof.finalize_launches++;
    ws->prof.kernel_launches++;
    ws->prof.queries += batch;
    if (ws->pending.size() > 4096) drain_events(ws, s);
    return DAWN_OK;
}

// int8 corpus, large batch, fp16-tile variant: chunk by chunk through a dequantised fp16 scratch (i8_tensor.cu),
// then one finalize over the gathered per-chunk lists with the exact int8 re-score.  Kept as the A/B partner of
// the native kind::i8 kernel ("i8_native" = 0).
constexpr float kI8DequantSlack = 5.6e-4f;  // |q.(fp16(s x8) - s x8)| <= 2^-11 ||q|| ||s x8||, plus a larger ||x~|| in the query-rounding term
int search_i8_tensor(dawn_index *idx, SearchWs *ws, const float *d_queries, size_t batch, size_t k, int kprime,
                     uint64_t *d_labels_out, float *d_dist_out, uint32_t *d_counts, uint32_t *d_flags, cudaStream_t s,
                     uint32_t *d_status_out) {
    const int kp = kprime < 64 ? 64 : kprime;  // more slack: the certificate has to absorb the dequantisation rounding
    const size_t n = ws->n_rows;
    const size_t want = (size_t)idx->i8_tensor_chunk_rows;
    const size_t n_chunks = (n + want - 1) / want;
    const size_t rpc = ((n + n_chunks - 1) / n_chunks + 255) / 256 * 256;  // rows per chunk, whole tiles
    const size_t qp = (batch + 255) / 256 * 256;
    int rc;
    if (rpc > ws->i8_scratch_rows) {
        if (ws->d_i8_scratch) cudaFree(ws->d_i8_scratch);
        ws->d_i8_scratch = nullptr;
        ws->i8_scratch_rows = 0;
        CK(idx, cudaMalloc(&ws->d_i8_scratch, rpc * (size_t)kRowBytesF16));
        ws->i8_scratch_rows = rpc;
    }
    if ((rc = ensure_dev(idx, &ws->d_i8_lists, &ws->i8_lists_cap, batch * n_chunks * kp))) return rc;
    if ((rc = ensure_dev(idx, &ws->d_i8_overflow, &ws->i8_overflow_cap, batch))) return rc;
    if ((rc = ensure_gemm_ws(idx, ws, gemm_workspace_bytes((int)batch)))) return rc;
    if ((rc = ensure_dev(idx, &ws->d_partials, &ws->partials_cap, qp * kp))) return rc;
    if ((rc = prepare_counters(idx, ws, 1, s))) return rc;
    CK(idx, cudaMemsetAsync(ws->d_i8_overflow, 0, batch * sizeof(uint32_t), s));
    const float *eps_q = nullptr;
    EventPair evg;
    bool timedg = begin_event(idx, ws, 2, s, &evg);
    for (size_t c = 0; c < n_chunks; c++) {
        const size_t base = c * rpc;
        const size_t rows = n - base < rpc ? n - base : rpc;
        CK(idx, launch_dequant_i8_f16(arena_i8(idx), base, rows, ws->d_i8_scratch, s));
        GemmSearch gs{};
        gs.corpus = ws->d_i8_scratch;
        gs.labels = idx->labels + base;
        gs.n_rows = rows;
        gs.queries = d_queries;
        gs.n_queries = (int)batch;
        gs.kprime = kp;
        fill_gemm_knobs(idx, gs);
        gs.workspace = ws->d_gemm_ws;
        gs.final_lists = ws->d_partials;
        gs.accum_slack = kGemmAccumSlack + kI8DequantSlack;
        gs.limit_score = -INFINITY;
        const uint32_t *overflow = nullptr;
        int launches = 0;
        gs.eps_out = &eps_q;
        gs.overflow_out = &overflow;
        gs.launches_out = &launches;
        CK(idx, launch_gemm_search(gs, s));
        CK(idx, launch_gather_chunk_lists(ws->d_partials, (int)batch, kp, (uint32_t)base, (int)c, (int)n_chunks, ws->d_i8_lists,
                                          overflow, ws->d_i8_overflow, s));
        ws->prof.gemm_batches++;
        ws->prof.kernel_launches += launches + 2;
    }
    if (timedg) end_event(ws, evg, s);
    FinalizeLaunch fl{};
    fl.corpus = idx->corpus;
    fl.queries = d_queries;
    fl.nq = (int)batch;
    fl.partials = ws->d_i8_lists;
    fl.n_lists = (int)n_chunks;
    fl.kprime = kp;
    fl.k = (int)k;
    fl.eps = 0.f;
    fl.labels_out = d_labels_out;
    fl.distances_out = d_dist_out;
    fl.counts_out = d_counts;
    fl.flags_out = d_flags;
    fl.scalar = 1;
    fl.eps_q = eps_q;  // same queries and slack for every chunk: the last chunk's values are everybody's
    fl.overflow = ws->d_i8_overflow;
    fl.counters = ws->d_counters;
    fl.n_counters = 1;
    fl.status_out = d_status_out;
    return run_finalize(idx, ws, fl, s, batch);
}

// int8 corpus, large batch, native variant (gemm_i8.cu): tcgen05 kind::i8 straight from the int8 arena; the rounds leave
// the k' best rows by EXACT score, finalize orders them.
int search_i8_native(dawn_index *idx, SearchWs *ws, const float *d_queries, size_t batch, size_t k, int kprime,
                     uint64_t *d_labels_out, float *d_dist_out, uint32_t *d_counts, uint32_t *d_flags, cudaStream_t s,
                     uint32_t *d_status_out) {
    const size_t qp = (batch + 255) / 256 * 256;
    int rc;
    // The rounds rank EXACT scores, so no slack is needed for the certificate beyond "the k'-th is strictly worse than
    // the k-th": k' = k + 4 (rounded up to 4, at least 16) instead of the scan paths' 16/32/64/128 -- fewer survivors per
    // round to log and re-score (k = 100: 104 instead of 128).
    {
        int kp = ((int)k + 4 + 3) / 4 * 4;
        if (kp < 16) kp = 16;
        if (kp < kprime) kprime = kp;
    }
    if ((rc = ensure_gemm_ws(idx, ws, gemm_i8_workspace_bytes((int)batch)))) return rc;
    if ((rc = ensure_dev(idx, &ws->d_partials, &ws->partials_cap, qp * kprime))) return rc;
    if ((rc = prepare_counters(idx, ws, 1, s))) return rc;
    GemmSearchI8 gs{};
    gs.arena = arena_i8(idx);
    gs.labels = idx->labels;
    gs.n_rows = ws->n_rows;
    gs.queries = d_queries;
    gs.n_queries = (int)batch;
    gs.kprime = kprime;
    gs.grid = idx->sm_count;
    gs.cta_group = (int)idx->gemm_cta_group;
    gs.chunk_tiles = (int)idx->gemm_chunk_tiles;
    gs.sequential_tiles = (int)idx->gemm_sequential_tiles;
    gs.growth = (int)idx->gemm_growth;
    gs.no_unit_sync = idx->gemm_unit_sync ? 0 : 1;
    gs.workspace = ws->d_gemm_ws;
    gs.final_lists = ws->d_partials;
    gs.limit_score = ws->eps_scale == 1.0f ? ws->limit_score : -INFINITY;
    gs.eps_scale = ws->eps_scale;
    const uint32_t *overflow = nullptr;
    int launches = 0;
    gs.overflow_out = &overflow;
    gs.launches_out = &launches;
    EventPair evg;
    bool timedg = begin_event(idx, ws, 2, s, &evg);
    CK(idx, launch_gemm_search_i8(gs, s));
    if (timedg) end_event(ws, evg, s);
    ws->prof.gemm_batches++;
    ws->prof.kernel_launches += launches;
    FinalizeLaunch fl{};
    fl.corpus = idx->corpus;
    fl.queries = d_queries;
    fl.nq = (int)batch;
    fl.partials = ws->d_partials;
    fl.n_lists = 1;
    fl.kprime = kprime;
    fl.k = (int)k;
    fl.eps = 0.f;  // the candidates carry exact scores: a row outside the list scores strictly below its weakest member
    fl.labels_out = d_labels_out;
    fl.distances_out = d_dist_out;
    fl.counts_out = d_counts;
    fl.flags_out = d_flags;
    fl.scalar = 1;
    fl.eps_q = nullptr;
    fl.overflow = overflow;
    fl.counters = ws->d_counters;
    fl.n_counters = 1;
    fl.status_out = d_status_out;
    return run_finalize(idx, ws, fl, s, batch);
}

// fp16 corpus with an int8 shadow (option "shadow_i8"): the rounds FILTER on the shadow with the int8 tensor cores (half the
// bytes and twice the MMA rate of the fp16 tiles) and rank the survivors by their exact score over the fp16 rows, so the
// rounds leave the k' best rows by EXACT score and finalize -- the same fp16 re-score as every other path -- orders them.
int search_f16_shadow(dawn_index *idx, SearchWs *ws, const uint8_t *shadow, float kappa, const float *d_queries, size_t batch,
                      size_t k, int kprime, uint64_t *d_labels_out, float *d_dist_out, uint32_t *d_counts, uint32_t *d_flags,
                      cudaStream_t s, uint32_t *d_status_out) {
    const size_t qp = (batch + 255) / 256 * 256;
    int rc;
    {
        int kp = ((int)k + 4 + 3) / 4 * 4;  // exact scores are ranked: k' = k + 4 is all the certificate needs (see search_i8_native)
        if (kp < 16) kp = 16;
        if (kp < kprime) kprime = kp;
    }
    if ((rc = ensure_gemm_ws(idx, ws, gemm_i8_workspace_bytes((int)batch)))) return rc;
    if ((rc = ensure_dev(idx, &ws->d_partials, &ws->partials_cap, qp * kprime))) return rc;
    if ((rc = prepare_counters(idx, ws, 1, s))) return rc;
    GemmSearchI8 gs{};
    gs.arena = shadow;
    gs.labels = idx->labels;
    gs.n_rows = ws->n_rows;
    gs.queries = d_queries;
    gs.n_queries = (int)batch;
    gs.kprime = kprime;
    gs.grid = idx->sm_count;
    gs.cta_group = (int)idx->gemm_cta_group;
    gs.chunk_tiles = (int)idx->gemm_chunk_tiles;
    gs.sequential_tiles = (int)idx->gemm_sequential_tiles;
    gs.growth = (int)idx->gemm_growth;
    gs.no_unit_sync = idx->gemm_unit_sync ? 0 : 1;
    gs.workspace = ws->d_gemm_ws;
    gs.final_lists = ws->d_partials;
    gs.limit_score = ws->limit_score;
    gs.eps_scale = 1.0f;
    gs.rescore_f16 = idx->corpus;
    gs.shadow_kappa = kappa;
    const uint32_t *overflow = nullptr;
    int launches = 0;
    gs.overflow_out = &overflow;
    gs.launches_out = &launches;
    EventPair evg;
    bool timedg = begin_event(idx, ws, 2, s, &evg);
    CK(idx, launch_gemm_search_i8(gs, s));
    if (timedg) end_event(ws, evg, s);
    ws->prof.gemm_batches++;
    ws->prof.shadow_batches++;
    ws->prof.kernel_launches += launches;
    FinalizeLaunch fl{};
    fl.corpus = idx->corpus;
    fl.queries = d_queries;
    fl.nq = (int)batch;
    fl.partials = ws->d_partials;
    fl.n_lists = 1;
    fl.kprime = kprime;
    fl.k = (int)k;
    fl.eps = 0.f;  // the candidates carry exact scores: a row outside the list scores strictly below its weakest member
    fl.labels_out = d_labels_out;
    fl.distances_out = d_dist_out;
    fl.counts_out = d_counts;
    fl.flags_out = d_flags;
    fl.scalar = 0;
    fl.eps_q = nullptr;
    fl.overflow = overflow;
    fl.counters = ws->d_counters;
    fl.n_counters = 1;
    fl.status_out = d_status_out;
    return run_finalize(idx, ws, fl, s, batch);
}

// Enqueue the whole search for `batch` device-resident queries on stream `s`.  The caller holds the shared
// corpus lock; ws->n_rows / eps_scale / limit_score describe the snapshot being searched.
int search_enqueue(dawn_index *idx, SearchWs *ws, const float *d_queries, size_t batch, size_t k, int kprime,
                   uint64_t *d_labels_out, float *d_dist_out, uint32_t *d_counts, uint32_t *d_flags,
                   cudaStream_t s, bool scan_only = false, uint32_t *d_status_out = nullptr) {
    const int grid = idx->sm_count;
    const size_t n = ws->n_rows;
    int rc;
    // a pushed-down limit is only sound with the nominal eps values
    const float limit_score = ws->eps_scale == 1.0f ? ws->limit_score : -INFINITY;
    // DAWN_SCALAR_F32: candidates are selected on the fp16 copies and re-scored on the f32 vectors as given; the copies'
    // rounding (<= kF32StoreSlack in score) joins every eps, and the lists are at least 64 deep so the certificate has room
    const bool f32_store = idx->scalar == DAWN_SCALAR_F32;
    const float store_slack = f32_store ? kF32StoreSlack : 0.0f;
    if (f32_store && kprime < 64) kprime = 64;
    const bool i8_small_on_big = (int64_t)batch >= idx->gemm_small_batch && (int64_t)n >= idx->gemm_small_batch_rows;
    // A row with an inf or NaN component (or, in an fp16 copy, one at +-65504) breaks the tensor-core paths and the shadow: an
    // fp16 query component below 2^-25 is 0 there and 0 * inf is NaN, and the shadow stores such a row as zeros.  The scan
    // multiplies by the f32 query, in the order the oracle does, so it alone answers such an index.
    if (ws->odd_rows) scan_only = true;
    if (idx->scalar == DAWN_SCALAR_I8 && !scan_only && idx->i8_tensor_min_batch > 0 &&
        ((int64_t)batch >= idx->i8_tensor_min_batch || i8_small_on_big) && n >= 65536 && idx->i8_native)
        return search_i8_native(idx, ws, d_queries, batch, k, kprime, d_labels_out, d_dist_out, d_counts, d_flags, s, d_status_out);
    if (idx->scalar == DAWN_SCALAR_I8 && !scan_only && idx->i8_tensor_min_batch > 0 &&
        (int64_t)batch >= idx->i8_tensor_min_batch && n >= 65536 && k <= 100)
        return search_i8_tensor(idx, ws, d_queries, batch, k, kprime, d_labels_out, d_dist_out, d_counts, d_flags, s, d_status_out);
    if (idx->scalar == DAWN_SCALAR_I8) {
        // K4: int8 storage -> streaming dp4a scan, 1 or 2 queries per pass, exact f32 re-score
        const size_t need_ws = batch * (sizeof(I8Query) + sizeof(float)) + 256;
        if ((rc = ensure_gemm_ws(idx, ws, need_ws))) return rc;
        I8Query *d_iq = static_cast<I8Query *>(ws->d_gemm_ws);
        float *d_eps = reinterpret_cast<float *>(static_cast<uint8_t *>(ws->d_gemm_ws) + batch * sizeof(I8Query));
        if ((rc = ensure_dev(idx, &ws->d_partials, &ws->partials_cap, batch * (size_t)grid * kprime))) return rc;
        const size_t need_counters = batch + 1;
        if ((rc = prepare_counters(idx, ws, need_counters, s))) return rc;
        CK(idx, launch_prep_queries_i8(d_queries, (int)batch, d_iq, d_eps, s));
        ws->prof.kernel_launches++;
        size_t done = 0, pass = 0;
        while (done < batch) {
            const int qt = batch - done >= 2 ? 2 : 1;
            ScanLaunchI8 sl;
            sl.corpus = arena_i8(idx);
            sl.labels = idx->labels;
            sl.n_rows = (uint32_t)n;
            sl.queries = d_iq + done;
            sl.nq = qt;
            sl.kprime = kprime;
            sl.partials = ws->d_partials + done * (size_t)grid * kprime;
            sl.chunk_counter = ws->d_counters + 1 + pass;
            sl.status = ws->d_counters;
            sl.grid = grid;
            sl.eps_q = d_eps + done;
            sl.limit_score = limit_score;
            EventPair ev;
            bool timed = begin_event(idx, ws, 0, s, &ev);
            CK(idx, launch_scan_topk_i8(sl, s));
            if (timed) end_event(ws, ev, s);
            ws->prof.scan_launches++;
            ws->prof.kernel_launches++;
            done += qt;
            pass++;
        }
        FinalizeLaunch fl{};
        fl.corpus = idx->corpus;
        fl.queries = d_queries;
        fl.nq = (int)batch;
        fl.partials = ws->d_partials;
        fl.n_lists = grid;
        fl.kprime = kprime;
        fl.k = (int)k;
        fl.eps = 0.f;
        fl.labels_out = d_labels_out;
        fl.distances_out = d_dist_out;
        fl.counts_out = d_counts;
        fl.flags_out = d_flags;
        fl.scalar = 1;
        fl.eps_q = d_eps;
        fl.overflow = nullptr;
        fl.counters = ws->d_counters;
        fl.n_counters = (int)need_counters;
        fl.status_out = d_status_out;
        return run_finalize(idx, ws, fl, s, batch);
    }
    const bool gemm_ok = n >= 1024 && batch >= 1;
    // the int8 shadow covers this snapshot (it is brought up to date before every search; rows are append-only)
    const uint8_t *shadow = nullptr;
    float kappa = 0.f;
    if (idx->scalar == DAWN_SCALAR_F16 && idx->shadow_i8 && ws->eps_scale == 1.0f && n >= 65536 && !scan_only && idx->force_path != 1) {
        shadow = idx->shadow.load();
        kappa = idx->shadow_kappa.load();
        if (!(shadow && idx->shadow_rows.load() >= n && kappa > 0.f)) shadow = nullptr;
    }
    const bool use_gemm = gemm_ok && !scan_only && idx->force_path != 1 &&
                          (idx->force_path == 2 ||
                           ((int64_t)batch >= idx->gemm_min_batch && (int64_t)n >= idx->gemm_min_rows) ||
                           ((int64_t)batch >= idx->gemm_small_batch && (int64_t)n >= idx->gemm_small_batch_rows) ||
                           // with a shadow even a single query over a big corpus is cheaper through the int8 rounds (388 B per
                           // row instead of the scan's 768 B; the rounds' fixed cost is ~0.25 ms): 10M rows 1.08 -> 0.85 ms,
                           // 100M rows 11.9 -> 6.1 ms (tools/shadow_batch1.py)
                           (shadow && (int64_t)n >= idx->shadow_single_rows));
    // A large k on a compute-bound batch over a small shard is the one case where the shadow loses: its wider filter band
    // times k' = k + 4 candidates makes the exact re-scores between rounds cost more than the int8 tiles save (12.5M rows,
    // 1024 queries, k = 100: 9.4 ms against 7.5 ms on the fp16 tiles; k = 20: 6.5 against 7.2; k = 10: 5.7 against 7.0).
    if (shadow && batch >= 128 && k > 32 && (int64_t)n < idx->shadow_big_k_rows) shadow = nullptr;
    if (use_gemm && shadow)
        return search_f16_shadow(idx, ws, shadow, kappa, d_queries, batch, k, kprime, d_labels_out, d_dist_out, d_counts, d_flags, s,
                                 d_status_out);
    if (use_gemm) {
        const size_t qp = (batch + 255) / 256 * 256;
        if ((rc = ensure_gemm_ws(idx, ws, gemm_workspace_bytes((int)batch)))) return rc;
        if ((rc = ensure_dev(idx, &ws->d_partials, &ws->partials_cap, qp * kprime))) return rc;
        if ((rc = prepare_counters(idx, ws, 1, s))) return rc;
        GemmSearch gs{};
        gs.corpus = idx->corpus;
        gs.labels = idx->labels;
        gs.n_rows = n;
        gs.queries = d_queries;
        gs.n_queries = (int)batch;
        gs.kprime = kprime;
        fill_gemm_knobs(idx, gs);
        gs.workspace = ws->d_gemm_ws;
        gs.final_lists = ws->d_partials;
        gs.accum_slack = kGemmAccumSlack + store_slack;
        gs.limit_score = limit_score > -INFINITY ? limit_score - store_slack : limit_score;
        const float *eps_q = nullptr;
        const uint32_t *overflow = nullptr;
        int launches = 0;
        gs.eps_out = &eps_q;
        gs.overflow_out = &overflow;
        gs.launches_out = &launches;
        EventPair evg;
        bool timedg = begin_event(idx, ws, 2, s, &evg);
        CK(idx, launch_gemm_search(gs, s));
        if (timedg) end_event(ws, evg, s);
        ws->prof.gemm_batches++;
        ws->prof.kernel_launches += launches;
        FinalizeLaunch fl{};
        fl.corpus = idx->corpus;
        fl.queries = d_queries;
        fl.nq = (int)batch;
        fl.partials = ws->d_partials;
        fl.n_lists = 1;
        fl.kprime = kprime;
        fl.k = (int)k;
        fl.eps = 0.f;
        fl.labels_out = d_labels_out;
        fl.distances_out = d_dist_out;
        fl.counts_out = d_counts;
        fl.flags_out = d_flags;
        fl.scalar = f32_store ? 2 : 0;
        fl.corpus32 = idx->corpus32;
        fl.eps_q = eps_q;
        fl.overflow = overflow;
        fl.counters = ws->d_counters;
        fl.n_counters = 1;
        fl.status_out = d_status_out;
        return run_finalize(idx, ws, fl, s, batch);
    }
    if ((rc = ensure_dev(idx, &ws->d_partials, &ws->partials_cap, batch * (size_t)grid * kprime))) return rc;
    const size_t need_counters = batch + 1;
    if ((rc = prepare_counters(idx, ws, need_counters, s))) return rc;

    size_t done = 0;
    size_t pass = 0;
    const int max_qt = scan_max_queries_per_pass(kprime);
    while (done < batch) {
        size_t left = batch - done;
        int qt = left >= 4 && max_qt >= 4 ? 4 : (left >= 2 && max_qt >= 2 ? 2 : 1);
        ScanLaunch sl;
        sl.corpus = idx->corpus;
        sl.labels = idx->labels;
        sl.n_rows = (uint32_t)n;
        sl.queries = d_queries + done * kDim;
        sl.nq = qt;
        sl.kprime = kprime;
        sl.partials = ws->d_partials + done * (size_t)grid * kprime;
        sl.chunk_counter = ws->d_counters + 1 + pass;
        sl.status = ws->d_counters;
        sl.grid = grid;
        // no pushed-down limit: the scan's error grows with |q|, which the host does not know for device-resident queries, so
        // a floor of limit_score - 2 eps dropped hits of long queries (limit applied afterwards, by the callers)
        sl.score_floor = -INFINITY;
        EventPair ev;
        bool timed = begin_event(idx, ws, 0, s, &ev);
        CK(idx, launch_scan_topk_f16(sl, s));
        if (timed) end_event(ws, ev, s);
        debug_wait(ws, s, "scan_topk_f16");
        ws->prof.scan_launches++;
        ws->prof.kernel_launches++;
        done += qt;
        pass++;
    }
    FinalizeLaunch fl{};
    fl.corpus = idx->corpus;
    fl.queries = d_queries;
    fl.nq = (int)batch;
    fl.partials = ws->d_partials;
    fl.n_lists = grid;
    fl.kprime = kprime;
    fl.k = (int)k;
    fl.eps = kScanEps + store_slack;
    fl.labels_out = d_labels_out;
    fl.distances_out = d_dist_out;
    fl.counts_out = d_counts;
    fl.flags_out = d_flags;
    fl.scalar = f32_store ? 2 : 0;
    fl.corpus32 = idx->corpus32;
    fl.eps_q = nullptr;
    fl.overflow = nullptr;
    fl.counters = ws->d_counters;
    fl.n_counters = (int)need_counters;
    fl.status_out = d_status_out;
    if (debug_stages())
        fprintf(stderr, "[dawn debug] finalize: nq %d lists %d k' %d k %d out %p\n", fl.nq, fl.n_lists, fl.kprime, fl.k,
                (void *)fl.labels_out);
    rc = run_finalize(idx, ws, fl, s, batch);
    debug_wait(ws, s, "finalize (scan path)");
    return rc;
}

// Snapshot the searchable state: flush staged adds, run the norm gate over new rows, take the shared corpus lock.
int snapshot_for_search(dawn_index *idx, std::shared_lock<std::shared_mutex> &rd, size_t *n_rows, float *eps_scale,
                        bool *odd_rows = nullptr) {
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = flush_staged(idx);
    if (rc) return rc;
    rc = ensure_norms_checked(idx);
    if (rc) return rc;
    rc = ensure_shadow(idx);
    if (rc) return rc;
    *n_rows = idx->size;
    *eps_scale = eps_scale_of(idx);
    if (odd_rows) *odd_rows = idx->odd_rows != 0;
    rd = std::shared_lock<std::shared_mutex>(idx->corpus_mu);
    return DAWN_OK;
}

int search_batch_host(dawn_index *idx, const float *queries, size_t batch, size_t k, float distance_limit,
                      uint64_t *labels_out, float *distances_out, size_t *counts_out) {
    int rc = check_alive(idx);
    if (rc) return rc;
    if (batch == 0) return DAWN_OK;
    if (!queries || !counts_out) return fail(DAWN_ERR_INVALID, "queries / counts_out is null");
    if (k > DAWN_MAX_K) return fail(DAWN_ERR_INVALID, "k = %zu exceeds DAWN_MAX_K = %d", k, DAWN_MAX_K);
    if (k > 0 && (!labels_out || !distances_out)) return fail(DAWN_ERR_INVALID, "output buffer is null");
    std::shared_lock<std::shared_mutex> rd;
    size_t n = 0;
    float eps_scale = 1.0f;
    bool odd_rows = false;
    rc = snapshot_for_search(idx, rd, &n, &eps_scale, &odd_rows);
    if (rc) return rc;
    if (k == 0 || n == 0) {
        for (size_t b = 0; b < batch; b++) counts_out[b] = 0;
        return DAWN_OK;
    }
    WsLease lease(idx);
    SearchWs *ws = lease.ws;
    if (!ws) return fail(DAWN_ERR_CUDA, "cannot create a search workspace (stream / event creation failed)");
    ws->n_rows = n;
    ws->eps_scale = eps_scale;
    ws->odd_rows = odd_rows;
    ws->limit_score = (distance_limit == distance_limit && distance_limit < INFINITY) ? (float)(1.0 - (double)distance_limit)
                                                                                      : -INFINITY;
    rc = ensure_query_ws(idx, ws, batch, k);
    if (rc) return rc;
    cudaStream_t s = ws->stream;
    memcpy(ws->h_queries, queries, batch * kDim * sizeof(float));
    CK(idx, cudaMemcpyAsync(ws->d_queries, ws->h_queries, batch * kDim * sizeof(float), cudaMemcpyHostToDevice, s));
    int kprime = choose_kprime(k);
    const uint64_t gemm_before = ws->prof.gemm_batches;
    ResultView dv = result_view(ws->d_result, batch, k), hv = result_view(ws->h_result, batch, k);
    // A small result block is written by the finalize kernel straight into the pinned host buffer (it is
    // device-accessible under unified addressing): a few hundred bytes of posted PCIe writes instead of a
    // copy-engine round trip after the kernel.  Large blocks go through one D2H copy.
    const bool direct = dv.bytes <= kDirectResultBytes && !getenv("DAWN_NO_DIRECT_RESULT");
    const ResultView &ov = direct ? hv : dv;
    rc = search_enqueue(idx, ws, ws->d_queries, batch, k, kprime, ov.labels, ov.dist, ov.counts, ov.flags, s, false, ov.status);
    if (rc) return rc;
    ws->counters_clean = true;  // every path ends with a finalize that zeroes the counters it used
    if (!direct) CK(idx, cudaMemcpyAsync(ws->h_result, ws->d_result, dv.bytes, cudaMemcpyDeviceToHost, s));  // the one D2H
    CK(idx, cudaStreamSynchronize(s));
    if (hv.status[0] != 0) return fail(DAWN_ERR_INTERNAL, "scan kernel reported status 0x%x", hv.status[0]);
    memcpy(labels_out, hv.labels, batch * k * sizeof(uint64_t));
    memcpy(distances_out, hv.dist, batch * k * sizeof(float));
    for (size_t b = 0; b < batch; b++) counts_out[b] = hv.counts[b];

    // Exactness certificate not met (near-ties deeper than the slack, or a tensor-core-path log
    // overflow): re-run those queries through the f32 scan with the longest candidate list.
    const bool can_escalate = kprime < kMaxCand || ws->prof.gemm_batches > gemm_before;
    std::vector<size_t> redo;
    for (size_t b = 0; b < batch; b++)
        if (!(hv.flags[b] & 1u)) redo.push_back(b);
    if (!can_escalate) {
        ws->prof.uncertified += redo.size();
        return DAWN_OK;
    }
    for (size_t b : redo) {
        ws->prof.escalations++;
        ResultView d1 = result_view(ws->d_result, 1, k), h1 = result_view(ws->h_result, 1, k);
        const bool direct1 = d1.bytes <= kDirectResultBytes;
        const ResultView &o1 = direct1 ? h1 : d1;
        rc = search_enqueue(idx, ws, ws->d_queries + b * kDim, 1, k, kMaxCand, o1.labels, o1.dist, o1.counts, o1.flags, s,
                            /*scan_only=*/true, o1.status);
        if (rc) return rc;
        ws->counters_clean = true;
        if (!direct1) CK(idx, cudaMemcpyAsync(ws->h_result, ws->d_result, d1.bytes, cudaMemcpyDeviceToHost, s));
        CK(idx, cudaStreamSynchronize(s));
        memcpy(labels_out + b * k, h1.labels, k * sizeof(uint64_t));
        memcpy(distances_out + b * k, h1.dist, k * sizeof(float));
        counts_out[b] = h1.counts[0];
        if (!(h1.flags[0] & 1u)) ws->prof.uncertified++;
    }
    return DAWN_OK;
}

// ---- bulk load pipeline -----------------------------------------------------------------------
// A large add_batch is cut into 8192-row slices dealt round-robin to kBulkThreads copier threads.  Each thread
// copies its slice into one of its two pinned buffers (the host-side memcpy is what limited the single-threaded
// path to ~12 GB/s), then enqueues H2D + K1 + labels on its own stream, so host copies, PCIe transfers and the
// conversion kernels of different slices overlap.  Row positions are fixed by the slice index, so the stored
// order equals the caller's order.

int bulk_setup(dawn_index *idx) {
    if (idx->bulk_ready) return DAWN_OK;
    for (int t = 0; t < kBulkThreads; t++) {
        BulkLane &L = idx->bulk[t];
        CK(idx, cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking));
        for (int b = 0; b < 2; b++) {
            CK(idx, cudaMallocHost(&L.h_buf[b], kStageRowsHost * kDim * sizeof(float)));
            CK(idx, cudaMallocHost(&L.h_lab[b], kStageRowsHost * sizeof(uint64_t)));
            CK(idx, cudaMalloc(&L.d_buf[b], kStageRowsHost * kDim * sizeof(float)));
            CK(idx, cudaEventCreateWithFlags(&L.done[b], cudaEventDisableTiming));
        }
    }
    idx->bulk_ready = true;
    return DAWN_OK;
}

void bulk_teardown(dawn_index *idx) {
    for (int t = 0; t < kBulkThreads; t++) {
        BulkLane &L = idx->bulk[t];
        if (L.stream) cudaStreamSynchronize(L.stream);
        for (int b = 0; b < 2; b++) {
            cudaFreeHost(L.h_buf[b]);
            cudaFreeHost(L.h_lab[b]);
            cudaFree(L.d_buf[b]);
            if (L.done[b]) cudaEventDestroy(L.done[b]);
        }
        if (L.stream) cudaStreamDestroy(L.stream);
    }
}

// idx->mu held; nothing staged.  Appends n rows starting at idx->size.
int bulk_add(dawn_index *idx, const uint64_t *labels, const float *vectors, size_t n) {
    int rc = bulk_setup(idx);
    if (rc) return rc;
    const size_t at = idx->size;
    const size_t n_slices = (n + kStageRowsHost - 1) / kStageRowsHost;
    static const int lanes = [] {
        const char *e = getenv("DAWN_BULK_THREADS");
        int v = e ? atoi(e) : 8;
        return v < 1 ? 1 : (v > kBulkThreads ? kBulkThreads : v);
    }();
    std::atomic<int> err{0};
    auto lane_fn = [&](int t) {
        cudaSetDevice(idx->device);
        BulkLane &L = idx->bulk[t];
        int turn = 0;
        for (size_t sl = (size_t)t; sl < n_slices && !err; sl += lanes, turn ^= 1) {
            const size_t r0 = sl * kStageRowsHost;
            const size_t cnt = n - r0 < kStageRowsHost ? n - r0 : kStageRowsHost;
            if (L.busy[turn]) {
                if (cudaEventSynchronize(L.done[turn]) != cudaSuccess) { err = 1; break; }
                L.busy[turn] = false;
            }
            memcpy(L.h_buf[turn], vectors + r0 * kDim, cnt * kDim * sizeof(float));
            memcpy(L.h_lab[turn], labels + r0, cnt * sizeof(uint64_t));
            cudaError_t e = cudaMemcpyAsync(L.d_buf[turn], L.h_buf[turn], cnt * kDim * sizeof(float), cudaMemcpyHostToDevice, L.stream);
            if (e == cudaSuccess)
                e = idx->scalar == DAWN_SCALAR_I8 ? launch_ingest_i8(L.d_buf[turn], arena_i8(idx), at + r0, cnt, L.stream)
                                                  : launch_ingest_f16(L.d_buf[turn], idx->corpus + (at + r0) * kDim, cnt, L.stream,
                                                                      idx->corpus32 != nullptr);
            if (e == cudaSuccess && idx->corpus32)
                e = cudaMemcpyAsync(idx->corpus32 + (at + r0) * kDim, L.d_buf[turn], cnt * kDim * sizeof(float), cudaMemcpyDeviceToDevice, L.stream);
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(idx->labels + at + r0, L.h_lab[turn], cnt * sizeof(uint64_t), cudaMemcpyHostToDevice, L.stream);
            if (e == cudaSuccess) e = cudaEventRecord(L.done[turn], L.stream);
            if (e != cudaSuccess) { err = 1; break; }
            L.busy[turn] = true;
        }
        if (cudaStreamSynchronize(L.stream) != cudaSuccess) err = 1;
        L.busy[0] = L.busy[1] = false;
    };
    std::thread th[kBulkThreads];
    for (int t = 1; t < lanes; t++) th[t] = std::thread(lane_fn, t);
    lane_fn(0);
    for (int t = 1; t < lanes; t++) th[t].join();
    if (err) {
        idx->dead = true;
        cudaError_t e = cudaGetLastError();
        return fail(DAWN_ERR_CUDA, "bulk add failed: %s", cudaGetErrorString(e));
    }
    idx->size = at + n;
    {
        std::lock_guard<std::mutex> lk(idx->prof_mu);
        idx->prof.kernel_launches += n_slices;
    }
    return DAWN_OK;
}

// ---- remove: compaction (remove.cu) ----------------------------------------------------------------
// idx->mu held.  Staged adds are flushed and every row is norm-checked and, when a shadow exists, quantised BEFORE the rows
// are paired: a donor moves below the new size, and a row that had not passed the gate scan or the quantiser by then would
// sit below both watermarks forever.  Mark and pair only read the label table, which nothing else writes while mu is held,
// so they run while searches go on; the moves and the new size are published under the exclusive corpus lock after every
// search in flight has finished, like a reallocation (grow_physical).
// A moved shadow row keeps its own scale: the kappa bound is per row, and the filter's chunk test takes the largest scale of
// the chunk's columns, so a 32-row group that receives a donor stays rigorous, only possibly looser -- like a group split by
// an append.  At most one group per removed row becomes mixed.  The norm statistics are left as they are: they bound a
// superset of the stored rows, so the certificate stays sound; dawn_index_verify rescans from zero and tightens them.
int remove_rows(dawn_index *idx, const uint64_t *req, size_t m, size_t *removed) {
    *removed = 0;
    int rc;
    if ((rc = flush_staged(idx)) || (rc = ensure_norms_checked(idx)) || (rc = ensure_shadow(idx))) return rc;
    const size_t n = idx->size;
    if (n == 0) return DAWN_OK;
    cudaStream_t s = idx->stream;
    const size_t req_bytes = (m * sizeof(uint64_t) + 255) / 256 * 256;
    uint8_t *scratch = nullptr;
    uint32_t *pairs = nullptr;
    const size_t scratch_bytes = req_bytes + remove_scratch_bytes(m, n);
    if (cudaMallocAsync(reinterpret_cast<void **>(&scratch), scratch_bytes, s) != cudaSuccess) {
        cudaGetLastError();
        return fail(DAWN_ERR_CAPACITY, "cannot allocate %zu bytes of HBM to remove %zu labels", scratch_bytes, m);
    }
    auto release = [&] {
        cudaFreeAsync(scratch, s);
        if (pairs) cudaFreeAsync(pairs, s);
    };
    uint32_t meta[2] = {0, 0};
    cudaError_t e = cudaMemcpyAsync(scratch, req, m * sizeof(uint64_t), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = launch_remove_mark(reinterpret_cast<const uint64_t *>(scratch), m, idx->labels, n, scratch + req_bytes, meta, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    const uint32_t r = meta[0], h = meta[1];
    if (e == cudaSuccess && h > 0) {
        if (cudaMallocAsync(reinterpret_cast<void **>(&pairs), 2 * (size_t)h * sizeof(uint32_t), s) != cudaSuccess) {
            cudaGetLastError();
            pairs = nullptr;
            release();
            return fail(DAWN_ERR_CAPACITY, "cannot allocate the %u row pairs of a remove", h);
        }
        e = launch_remove_pair(scratch + req_bytes, m, n, r, h, pairs, pairs + h, s);
    }
    if (e != cudaSuccess || r == 0) {
        release();
        CK(idx, e);
        return DAWN_OK;
    }
    {
        std::unique_lock<std::shared_mutex> wr(idx->corpus_mu);
        wait_device_searches(idx);
        // A shadow that lags the corpus (it is only extended from 65536 rows on, and not while the option is off) would hand
        // unquantised donor rows to holes below its watermark: drop it instead, the next search that wants it rebuilds it.
        if (idx->shadow.load() && idx->shadow_rows < n) drop_shadow(idx);
        RemoveMove mv;
        mv.holes = pairs;
        mv.donors = pairs ? pairs + h : nullptr;
        mv.n_pairs = h;
        mv.arena = reinterpret_cast<uint8_t *>(idx->corpus);
        mv.i8 = idx->scalar == DAWN_SCALAR_I8;
        mv.corpus32 = idx->corpus32;
        mv.shadow = idx->shadow.load();
        mv.labels = idx->labels;
        e = launch_remove_move(mv, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e == cudaSuccess) {
            const size_t left = n - r;
            idx->size = left;
            if (idx->shadow_rows > left) idx->shadow_rows = left;
            if (idx->norm_checked > left) idx->norm_checked = left;
        }
    }
    release();
    CK(idx, e);
    {
        std::lock_guard<std::mutex> lk(idx->prof_mu);
        idx->prof.kernel_launches += h > 0 ? 5 : 3;
    }
    *removed = r;
    return DAWN_OK;
}

}  // namespace

// ------------------------------------------------------------------------------ C ABI

extern "C" {

const char *dawn_last_error(void) { return g_last_error.c_str(); }
const char *dawn_version(void) { return "libdawn_b200 0.2.0 sm_100a"; }

int dawn_index_create(const dawn_options *opts, dawn_index **out) {
    if (!out) return fail(DAWN_ERR_INVALID, "out is null");
    *out = nullptr;
    dawn_options o{};
    if (opts) o = *opts;
    if (o.dimensions != 0 && o.dimensions != DAWN_DIMENSIONS)
        return fail(DAWN_ERR_INVALID, "dimensions must be %d (src/search/vector.rs:26), got %u",
                    DAWN_DIMENSIONS, o.dimensions);
    if (o.metric != DAWN_METRIC_IP) return fail(DAWN_ERR_INVALID, "only MetricKind::IP is supported");
    if (o.scalar != DAWN_SCALAR_F16 && o.scalar != DAWN_SCALAR_I8 && o.scalar != DAWN_SCALAR_F32)
        return fail(DAWN_ERR_INVALID, "scalar must be DAWN_SCALAR_F16, DAWN_SCALAR_I8 or DAWN_SCALAR_F32, got %u", o.scalar);
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return fail(DAWN_ERR_CUDA, "no CUDA device available (%s); libdawn_b200 has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (o.device < 0 || o.device >= n_dev)
        return fail(DAWN_ERR_INVALID, "device %d out of range (found %d devices)", o.device, n_dev);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, o.device);
    if (e != cudaSuccess) return fail(DAWN_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(DAWN_ERR_CUDA, "device %d is sm_%d%d; libdawn_b200 is built for sm_100a only", o.device,
                    prop.major, prop.minor);
    dawn_index *idx = new (std::nothrow) dawn_index();
    if (!idx) return fail(DAWN_ERR_INTERNAL, "out of host memory");
    idx->device = o.device;
    idx->scalar = (int)o.scalar;
    idx->sm_count = prop.multiProcessorCount;
    int rc = DAWN_OK;
    do {
        if ((e = cudaSetDevice(o.device)) != cudaSuccess) break;
        if ((e = cudaStreamCreateWithFlags(&idx->stream, cudaStreamNonBlocking)) != cudaSuccess) break;
        for (int b = 0; b < 2 && e == cudaSuccess; b++) {
            if ((e = cudaMallocHost(&idx->h_stage_buf[b], kStageRowsHost * kDim * sizeof(float))) != cudaSuccess) break;
            if ((e = cudaMallocHost(&idx->h_labels_buf[b], kStageRowsHost * sizeof(uint64_t))) != cudaSuccess) break;
            if ((e = cudaMalloc(&idx->d_stage_buf[b], kStageRowsHost * kDim * sizeof(float))) != cudaSuccess) break;
            if ((e = cudaEventCreateWithFlags(&idx->stage_done[b], cudaEventDisableTiming)) != cudaSuccess) break;
        }
        if (e != cudaSuccess) break;
        idx->h_stage = idx->h_stage_buf[0];
        idx->h_stage_labels = idx->h_labels_buf[0];
        idx->d_stage = idx->d_stage_buf[0];
        if ((e = cudaMalloc(&idx->d_norm_stats, 4 * sizeof(uint32_t))) != cudaSuccess) break;
        if ((e = cudaMallocHost(&idx->h_norm_stats, 4 * sizeof(uint32_t))) != cudaSuccess) break;
        if ((e = cudaMalloc(&idx->d_stats, 4 * sizeof(uint32_t))) != cudaSuccess) break;
        if ((e = cudaMallocHost(&idx->h_stats, 4 * sizeof(uint32_t))) != cudaSuccess) break;
        if ((e = cudaMemset(idx->d_stats, 0, 4 * sizeof(uint32_t))) != cudaSuccess) break;
        if ((e = cudaMemset(idx->d_norm_stats, 0, 4 * sizeof(uint32_t))) != cudaSuccess) break;
    } while (0);
    if (e == cudaSuccess) {
        idx->dev_ws = new_ws();
        if (!idx->dev_ws) e = cudaErrorMemoryAllocation;
    }
    if (e != cudaSuccess) {
        rc = fail(DAWN_ERR_CUDA, "index setup failed: %s", cudaGetErrorString(e));
        dawn_index_free(idx);
        return rc;
    }
    if (o.capacity > 0) {
        rc = grow_physical(idx, o.capacity);
        if (rc != DAWN_OK) {
            dawn_index_free(idx);
            return rc;
        }
        idx->capacity = o.capacity;
    }
    *out = idx;
    return DAWN_OK;
}

void dawn_index_free(dawn_index *idx) {
    if (!idx) return;
    cudaSetDevice(idx->device);
    if (idx->stream) cudaStreamSynchronize(idx->stream);
    for (SearchWs *ws : idx->pool_free) free_ws(ws);
    free_ws(idx->dev_ws);
    if (idx->bulk_ready) bulk_teardown(idx);
    cudaFree(idx->corpus);
    cudaFree(idx->corpus32);
    cudaFree(idx->shadow.load());
    cudaFree(idx->d_shadow_kappa);
    cudaFree(idx->labels);
    for (int b = 0; b < 2; b++) {
        cudaFree(idx->d_stage_buf[b]);
        cudaFreeHost(idx->h_stage_buf[b]);
        cudaFreeHost(idx->h_labels_buf[b]);
        if (idx->stage_done[b]) cudaEventDestroy(idx->stage_done[b]);
    }
    cudaFree(idx->d_norm_stats);
    cudaFreeHost(idx->h_norm_stats);
    cudaFree(idx->d_stats);
    cudaFreeHost(idx->h_stats);
    if (idx->stream) cudaStreamDestroy(idx->stream);
    cudaGetLastError();
    delete idx;
}

int dawn_index_reserve(dawn_index *idx, size_t n) {
    int rc = check_alive(idx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(idx->mu);
    if (n <= idx->capacity) return DAWN_OK;
    rc = flush_staged(idx);  // the copy into a new arena must include every row already handed over
    if (rc) return rc;
    rc = grow_physical(idx, n);
    if (rc) return rc;
    idx->capacity = n;
    return DAWN_OK;
}

int dawn_index_add_batch(dawn_index *idx, const uint64_t *labels, const float *vectors, size_t n) {
    int rc = check_alive(idx);
    if (rc) return rc;
    if (n == 0) return DAWN_OK;
    if (!labels || !vectors) return fail(DAWN_ERR_INVALID, "labels / vectors is null");
    std::lock_guard<std::mutex> lk(idx->mu);
    if (idx->size + idx->staged + n > idx->capacity)
        return fail(DAWN_ERR_CAPACITY, "add of %zu vectors exceeds capacity %zu (size %zu): reserve first", n,
                    idx->capacity.load(), idx->size + idx->staged);
    if (n >= kBulkMinRows) {
        rc = flush_staged(idx);
        if (rc) return rc;
        return bulk_add(idx, labels, vectors, n);
    }
    size_t done = 0;
    while (done < n) {
        size_t room = kStageRowsHost - idx->staged;
        size_t take = n - done < room ? n - done : room;
        memcpy(idx->h_stage + idx->staged * kDim, vectors + done * kDim, take * kDim * sizeof(float));
        memcpy(idx->h_stage_labels + idx->staged, labels + done, take * sizeof(uint64_t));
        idx->staged += take;
        done += take;
        if (idx->staged == kStageRowsHost) {
            rc = flush_staged_async(idx);  // the next chunk is copied on the host while this one moves
            if (rc) return rc;
        }
    }
    return DAWN_OK;
}

int dawn_index_add(dawn_index *idx, uint64_t label, const float *vector384) {
    return dawn_index_add_batch(idx, &label, vector384, 1);
}

int dawn_index_add_synthetic(dawn_index *idx, uint64_t seed, uint64_t first_row, size_t n) {
    int rc = check_alive(idx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(idx->mu);
    rc = flush_staged(idx);
    if (rc) return rc;
    const size_t at = idx->size;
    if (at + n > idx->capacity)
        return fail(DAWN_ERR_CAPACITY, "add of %zu vectors exceeds capacity %zu (size %zu): reserve first", n,
                    idx->capacity.load(), at);
    if (idx->scalar == DAWN_SCALAR_I8) CK(idx, launch_synth_i8(arena_i8(idx), at, seed, first_row, n, idx->stream));
    else if (idx->scalar == DAWN_SCALAR_F32) {
        CK(idx, launch_synth_f32(idx->corpus32 + at * kDim, seed, first_row, n, idx->stream));
        CK(idx, launch_ingest_f16(idx->corpus32 + at * kDim, idx->corpus + at * kDim, n, idx->stream, true));
    } else CK(idx, launch_synth_f16(idx->corpus + at * kDim, seed, first_row, n, idx->stream));
    CK(idx, launch_iota_labels(idx->labels + at, first_row + 1, n, idx->stream));  // labels = first_row + i + 1
    CK(idx, cudaStreamSynchronize(idx->stream));
    idx->size = at + n;
    {
        std::lock_guard<std::mutex> lp(idx->prof_mu);
        idx->prof.kernel_launches += 2;
    }
    return DAWN_OK;
}

// The rows of every listed label are compacted out of the device corpus (remove_rows); capacity is kept.
int dawn_index_remove_batch(dawn_index *idx, const uint64_t *labels, size_t n, size_t *removed_out) {
    if (removed_out) *removed_out = 0;
    if (!idx) return fail(DAWN_ERR_INVALID, "null index handle");
    if (n > 0 && !labels) return fail(DAWN_ERR_INVALID, "labels is null");
    int rc = check_alive(idx);
    if (rc) return rc;
    if (n == 0) return DAWN_OK;
    std::lock_guard<std::mutex> lk(idx->mu);
    size_t removed = 0;
    rc = remove_rows(idx, labels, n, &removed);
    if (rc) return rc;
    if (removed_out) *removed_out = removed;
    return DAWN_OK;
}

int dawn_index_remove(dawn_index *idx, uint64_t label, size_t *removed_out) {
    return dawn_index_remove_batch(idx, &label, 1, removed_out);
}

int dawn_index_search_batch(dawn_index *idx, const float *queries, size_t batch, size_t k,
                            uint64_t *labels_out, float *distances_out, size_t *counts_out) {
    return search_batch_host(idx, queries, batch, k, NAN, labels_out, distances_out, counts_out);
}

// (f3) distance_limit of UdpPacket::Search (/root/reference/src/net/udp_packets.rs:29-39): hits with
// distance >= limit are not returned (src/net/udp_service.rs:196-199).  Results are ascending, so the
// filter truncates; the limit is also pushed down into the kernels (scan paths: score floor; tensor-core
// path: initial threshold), so rows that cannot pass it are never appended, merged or re-scored.
// limit = +inf or NaN keeps everything.
int dawn_index_search_batch_limit(dawn_index *idx, const float *queries, size_t batch, size_t k, float distance_limit,
                                  uint64_t *labels_out, float *distances_out, size_t *counts_out) {
    int rc = search_batch_host(idx, queries, batch, k, distance_limit, labels_out, distances_out, counts_out);
    if (rc != DAWN_OK) return rc;
    if (distance_limit == distance_limit) {
        for (size_t b = 0; b < batch; b++) {
            size_t keep = 0;
            while (keep < counts_out[b] && distances_out[b * k + keep] < distance_limit) keep++;
            counts_out[b] = keep;
        }
    }
    return DAWN_OK;
}

int dawn_index_search_limit(dawn_index *idx, const float *query384, size_t k, float distance_limit,
                            uint64_t *labels_out, float *distances_out, size_t *count_out) {
    return dawn_index_search_batch_limit(idx, query384, 1, k, distance_limit, labels_out, distances_out, count_out);
}

int dawn_index_search(dawn_index *idx, const float *query384, size_t k, uint64_t *labels_out,
                      float *distances_out, size_t *count_out) {
    return dawn_index_search_batch(idx, query384, 1, k, labels_out, distances_out, count_out);
}

// (f3) on the device API: the limit is pushed down like in dawn_index_search_batch_limit, and the counts are cut on the
// device (results ascend, so the filter of udp_service.rs:196-199 truncates) -- what a sharded search needs before its merge.
int dawn_index_search_device_limit(dawn_index *idx, const float *d_queries, size_t batch, size_t k, float distance_limit,
                                   uint64_t *d_labels_out, float *d_distances_out, uint32_t *d_counts_out,
                                   uint32_t *d_flags_out, void *stream) {
    int rc = check_alive(idx);
    if (rc) return rc;
    if (batch == 0) return DAWN_OK;
    if (!d_queries || !d_labels_out || !d_distances_out || !d_counts_out || !d_flags_out)
        return fail(DAWN_ERR_INVALID, "null device pointer");
    if (k == 0 || k > DAWN_MAX_K) return fail(DAWN_ERR_INVALID, "k = %zu out of range 1..%d", k, DAWN_MAX_K);
    std::shared_lock<std::shared_mutex> rd;
    size_t n = 0;
    float eps_scale = 1.0f;
    bool odd_rows = false;
    rc = snapshot_for_search(idx, rd, &n, &eps_scale, &odd_rows);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(idx->dev_mu);
    SearchWs *ws = idx->dev_ws;
    cudaStream_t s = stream ? (cudaStream_t)stream : ws->stream;
    if (n == 0) {
        CK(idx, cudaMemsetAsync(d_counts_out, 0, batch * sizeof(uint32_t), s));
        CK(idx, cudaMemsetAsync(d_flags_out, 0x01, batch * sizeof(uint32_t), s));  // bit0: an empty shard's (empty) answer is exact
        return DAWN_OK;
    }
    const bool limited = distance_limit == distance_limit && distance_limit < INFINITY;
    ws->n_rows = n;
    ws->eps_scale = eps_scale;
    ws->odd_rows = odd_rows;
    ws->limit_score = limited ? (float)(1.0 - (double)distance_limit) : -INFINITY;
    // the workspace is shared by all device-API searches on this handle: a search enqueued on another
    // stream than the previous one first waits for it
    if (ws->ws_used && ws->ws_stream != s) CK(idx, cudaStreamWaitEvent(s, ws->ws_done, 0));
    rc = search_enqueue(idx, ws, d_queries, batch, k, choose_kprime(k), d_labels_out, d_distances_out, d_counts_out,
                        d_flags_out, s);
    if (rc == DAWN_OK && distance_limit == distance_limit)
        CK(idx, launch_truncate_by_limit(d_distances_out, d_counts_out, batch, k, distance_limit, s));
    if (rc == DAWN_OK) {
        CK(idx, cudaEventRecord(ws->ws_done, s));
        ws->ws_stream = s;
        ws->ws_used = true;
        ws->counters_clean = true;
    }
    return rc;
}

int dawn_index_search_device(dawn_index *idx, const float *d_queries, size_t batch, size_t k,
                             uint64_t *d_labels_out, float *d_distances_out, uint32_t *d_counts_out,
                             uint32_t *d_flags_out, void *stream) {
    return dawn_index_search_device_limit(idx, d_queries, batch, k, NAN, d_labels_out, d_distances_out, d_counts_out,
                                          d_flags_out, stream);
}

size_t dawn_index_size(const dawn_index *idx) { return idx ? idx->size + idx->staged : 0; }
size_t dawn_index_capacity(const dawn_index *idx) { return idx ? idx->capacity.load() : 0; }
size_t dawn_index_dimensions(const dawn_index *idx) { return idx ? DAWN_DIMENSIONS : 0; }

int dawn_index_get(dawn_index *idx, uint64_t label, float *vector384_out) {
    int rc = check_alive(idx);
    if (rc) return rc;
    if (!vector384_out) return fail(DAWN_ERR_INVALID, "output is null");
    std::shared_lock<std::shared_mutex> rd;
    size_t n = 0;
    float eps_scale;
    rc = snapshot_for_search(idx, rd, &n, &eps_scale);
    if (rc) return rc;
    if (n == 0) return fail(DAWN_ERR_INVALID, "label %llu not found", (unsigned long long)label);
    WsLease lease(idx);
    SearchWs *ws = lease.ws;
    if (!ws) return fail(DAWN_ERR_CUDA, "cannot create a search workspace");
    rc = ensure_query_ws(idx, ws, 1, 1);
    if (rc) return rc;
    cudaStream_t s = ws->stream;
    uint32_t *d_row = reinterpret_cast<uint32_t *>(ws->d_result);
    uint32_t *h_row = reinterpret_cast<uint32_t *>(ws->h_result);
    CK(idx, launch_find_label(idx->labels, n, label, d_row, s));
    ws->prof.kernel_launches++;
    CK(idx, cudaMemcpyAsync(h_row, d_row, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CK(idx, cudaStreamSynchronize(s));
    if (h_row[0] == kNoRow) return fail(DAWN_ERR_INVALID, "label %llu not found", (unsigned long long)label);
    if (idx->scalar == DAWN_SCALAR_I8) CK(idx, launch_gather_f32_i8(arena_i8(idx), d_row, 1, ws->d_queries, s));
    else if (idx->scalar == DAWN_SCALAR_F32)  // the vector exactly as it was added
        CK(idx, cudaMemcpyAsync(ws->d_queries, idx->corpus32 + (size_t)h_row[0] * kDim, kDim * sizeof(float), cudaMemcpyDeviceToDevice, s));
    else CK(idx, launch_gather_f32(idx->corpus, d_row, 1, ws->d_queries, s));
    ws->prof.kernel_launches++;
    CK(idx, cudaMemcpyAsync(ws->h_queries, ws->d_queries, kDim * sizeof(float), cudaMemcpyDeviceToHost, s));
    CK(idx, cudaStreamSynchronize(s));
    memcpy(vector384_out, ws->h_queries, kDim * sizeof(float));
    return DAWN_OK;
}

// SearchProvider::verify (/root/reference/src/search/search_provider.rs:289-327) over the DEVICE corpus: the
// reference scans every stored BLOB for len == 1536 and 0.99 < |v| < 1.01; the length is structural here, the
// norm gate runs as one HBM-bound pass over the stored (fp16 / int8-dequantised) rows.
int dawn_index_verify(dawn_index *idx, size_t *bad_rows_out, float *min_norm_out, float *max_norm_out) {
    int rc = check_alive(idx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(idx->mu);
    rc = flush_staged(idx);
    if (rc) return rc;
    reset_norm_stats(idx);  // a verify is a full scan, like the reference's
    rc = ensure_norms_checked(idx);
    if (rc) return rc;
    if (bad_rows_out) *bad_rows_out = (size_t)idx->bad_rows;
    if (min_norm_out) *min_norm_out = idx->size ? idx->norm_min : 0.f;
    if (max_norm_out) *max_norm_out = idx->norm_max;
    return DAWN_OK;
}

// ---- save / load: header, labels, stored rows (raw device layout) -------------------------
struct SaveHeader {
    char magic[8];  // "DAWNB200"
    uint32_t version, scalar, dims, reserved;
    uint64_t size;
};

int dawn_index_save(dawn_index *idx, const char *path) {
    int rc = check_alive(idx);
    if (rc) return rc;
    if (!path) return fail(DAWN_ERR_INVALID, "path is null");
    std::lock_guard<std::mutex> lk(idx->mu);
    rc = flush_staged(idx);
    if (rc) return rc;
    const size_t n = idx->size;
    if (idx->scalar == DAWN_SCALAR_I8 && n % kI8BlockRows) {
        // the last 8-row block is partly unused: zero its unused rows and scales so the file is deterministic
        const size_t blk_end = (n + kI8BlockRows - 1) / kI8BlockRows * kI8BlockRows;
        CK(idx, cudaMemsetAsync(arena_i8(idx) + i8_row_offset(n), 0, (blk_end - n) * kDim, idx->stream));
        CK(idx, cudaMemsetAsync(arena_i8(idx) + i8_scale_offset(n), 0, (blk_end - n) * 4, idx->stream));
    }
    std::string tmp = std::string(path) + ".tmp";
    FILE *f = fopen(tmp.c_str(), "wb");
    if (!f) return fail(DAWN_ERR_IO, "cannot open %s for writing", tmp.c_str());
    SaveHeader h{};
    memcpy(h.magic, "DAWNB200", 8);
    h.version = 1;
    h.scalar = (uint32_t)idx->scalar;
    h.dims = kDim;
    h.size = n;
    bool ok = fwrite(&h, sizeof h, 1, f) == 1;
    // stream device memory out through the two pinned staging buffers: the D2H of slice i+1 runs while
    // slice i is written to the file
    const size_t buf_bytes = kStageRowsHost * kDim * sizeof(float);
    auto dump = [&](const void *dptr, size_t bytes) -> int {
        size_t off = 0;
        int cur = 0;
        size_t in_flight = 0;
        if (bytes) {
            in_flight = bytes < buf_bytes ? bytes : buf_bytes;
            CK(idx, cudaMemcpyAsync(idx->h_stage_buf[0], dptr, in_flight, cudaMemcpyDeviceToHost, idx->stream));
        }
        while (ok && off < bytes) {
            CK(idx, cudaStreamSynchronize(idx->stream));
            const size_t have = in_flight;
            const size_t next_off = off + have;
            if (next_off < bytes) {
                in_flight = bytes - next_off < buf_bytes ? bytes - next_off : buf_bytes;
                CK(idx, cudaMemcpyAsync(idx->h_stage_buf[cur ^ 1], (const char *)dptr + next_off, in_flight, cudaMemcpyDeviceToHost,
                                        idx->stream));
            }
            ok = fwrite(idx->h_stage_buf[cur], 1, have, f) == have;
            off = next_off;
            cur ^= 1;
        }
        CK(idx, cudaStreamSynchronize(idx->stream));
        return DAWN_OK;
    };
    rc = dump(idx->labels, n * sizeof(uint64_t));
    if (rc == DAWN_OK)  // F32 storage persists the vectors as given; the fp16 selection copy is rebuilt on load
        rc = idx->scalar == DAWN_SCALAR_F32 ? dump(idx->corpus32, n * (size_t)kDim * sizeof(float)) : dump(idx->corpus, arena_bytes(idx, n));
    ok = (fclose(f) == 0) && ok;
    if (rc != DAWN_OK || !ok) {
        remove(tmp.c_str());
        return rc != DAWN_OK ? rc : fail(DAWN_ERR_IO, "short write to %s", tmp.c_str());
    }
    if (rename(tmp.c_str(), path) != 0) {
        remove(tmp.c_str());
        return fail(DAWN_ERR_IO, "cannot rename %s to %s", tmp.c_str(), path);
    }
    return DAWN_OK;
}

// Loads into a FRESH arena and swaps it in only when the whole file has arrived, so any failure
// (bad header, short file, read error, CUDA error) leaves the index exactly as it was -- the reference
// falls back to a rebuild when load fails (search_provider.rs:115-116).
int dawn_index_load(dawn_index *idx, const char *path) {
    int rc = check_alive(idx);
    if (rc) return rc;
    if (!path) return fail(DAWN_ERR_INVALID, "path is null");
    std::lock_guard<std::mutex> lk(idx->mu);
    rc = flush_staged(idx);  // staged adds belong to the old contents; they must not leak into the loaded ones
    if (rc) return rc;
    FILE *f = fopen(path, "rb");
    if (!f) return fail(DAWN_ERR_IO, "cannot open %s", path);
    SaveHeader h{};
    if (fread(&h, sizeof h, 1, f) != 1 || memcmp(h.magic, "DAWNB200", 8) != 0 || h.version != 1 ||
        h.scalar != (uint32_t)idx->scalar || h.dims != kDim) {
        fclose(f);
        return fail(DAWN_ERR_IO, "%s is not a libdawn_b200 index file with this index's storage type", path);
    }
    fseek(f, 0, SEEK_END);
    long long flen = ftell(f);
    const size_t payload = idx->scalar == DAWN_SCALAR_F32 ? (size_t)h.size * kDim * sizeof(float) : arena_bytes(idx, h.size);
    long long want = (long long)sizeof h + (long long)h.size * 8 + (long long)payload;
    if (flen != want) {
        fclose(f);
        return fail(DAWN_ERR_IO, "%s is truncated (%lld bytes, expected %lld)", path, flen, want);
    }
    fseek(f, sizeof h, SEEK_SET);
    if (h.size > 0xFFFFFFF0ull) {
        fclose(f);
        return fail(DAWN_ERR_INVALID, "%s holds more than 2^32 rows", path);
    }
    size_t rows_alloc = h.size > idx->capacity ? (size_t)h.size : idx->capacity.load();
    __half *nc = nullptr;
    uint64_t *nl = nullptr;
    float *n32 = nullptr;
    // An EMPTY index with room (the start-up case: reserve, then load) is filled in place -- nothing can be lost, and a
    // second arena next to a pre-reserved 100M-row one would not fit.  Otherwise: fresh arena, swap on success.
    const bool in_place = idx->size == 0 && idx->phys >= (size_t)h.size && idx->phys > 0;
    if (in_place) {
        std::unique_lock<std::shared_mutex> wr(idx->corpus_mu);  // no search may be reading the (empty) arena's pointers
        wait_device_searches(idx);
        nc = idx->corpus;
        nl = idx->labels;
        n32 = idx->corpus32;
        rows_alloc = idx->phys;
    } else if (rows_alloc > 0) {
        rc = alloc_arena(idx, rows_alloc, &nc, &nl, &n32);
        if (rc) {
            fclose(f);
            return rc;
        }
    }
    const size_t buf_bytes = kStageRowsHost * kDim * sizeof(float);
    bool ok = true;
    cudaError_t ce = cudaSuccess;
    // double-buffered: the file read of slice i+1 overlaps the H2D of slice i
    auto slurp = [&](void *dptr, size_t bytes) {
        size_t off = 0;
        int cur = 0;
        while (ok && ce == cudaSuccess && off < bytes) {
            const size_t take = bytes - off < buf_bytes ? bytes - off : buf_bytes;
            if (idx->stage_busy[cur]) {
                ce = cudaEventSynchronize(idx->stage_done[cur]);
                idx->stage_busy[cur] = false;
                if (ce != cudaSuccess) break;
            }
            ok = fread(idx->h_stage_buf[cur], 1, take, f) == take;
            if (!ok) break;
            ce = cudaMemcpyAsync((char *)dptr + off, idx->h_stage_buf[cur], take, cudaMemcpyHostToDevice, idx->stream);
            if (ce == cudaSuccess) ce = cudaEventRecord(idx->stage_done[cur], idx->stream);
            idx->stage_busy[cur] = true;
            off += take;
            cur ^= 1;
        }
    };
    slurp(nl, h.size * sizeof(uint64_t));
    if (idx->scalar == DAWN_SCALAR_F32) {
        slurp(n32, payload);
        if (ok && ce == cudaSuccess && h.size) ce = launch_ingest_f16(n32, nc, (size_t)h.size, idx->stream, true);  // rebuild the selection copy
    } else {
        slurp(nc, payload);
    }
    fclose(f);
    cudaError_t se = cudaStreamSynchronize(idx->stream);
    idx->stage_busy[0] = idx->stage_busy[1] = false;
    if (ce == cudaSuccess) ce = se;
    if (!ok || ce != cudaSuccess) {
        if (!in_place) {
            cudaFree(nc);
            cudaFree(nl);
            cudaFree(n32);
        }
        if (ce != cudaSuccess) {
            cudaGetLastError();
            return fail(DAWN_ERR_IO, "copy to the device failed while loading %s: %s (index unchanged)", path, cudaGetErrorString(ce));
        }
        return fail(DAWN_ERR_IO, "read error on %s (index unchanged)", path);
    }
    if (in_place) {
        idx->size = (size_t)h.size;
        if (idx->capacity < (size_t)h.size) idx->capacity = (size_t)h.size;
        reset_norm_stats(idx);
        return DAWN_OK;
    }
    __half *oc;
    uint64_t *ol;
    float *o32;
    {
        std::unique_lock<std::shared_mutex> wr(idx->corpus_mu);
        wait_device_searches(idx);
        oc = idx->corpus;
        ol = idx->labels;
        o32 = idx->corpus32;
        idx->corpus = nc;
        idx->labels = nl;
        idx->corpus32 = n32;
        idx->phys = rows_alloc;
        drop_shadow(idx);
        idx->size = (size_t)h.size;
        if (idx->capacity < (size_t)h.size) idx->capacity = (size_t)h.size;
    }
    cudaFree(oc);
    cudaFree(ol);
    cudaFree(o32);
    reset_norm_stats(idx);
    return DAWN_OK;
}

// ---- evidence for the certificate's constants (tests/test_gpu_slack.py) -----------------------------------
// Every (query,row) score the tensor cores produce for `batch` host queries against an index of <= 2048 rows is compared
// on the device with (a) the f64 dot product of the SAME fp16 operands (pure accumulation error of the MMA), (b) the
// sequential f32 re-score (what the exact answer is made of) and (c) the f64 dot product of the f32 query (the re-score's own
// rounding).  Results accumulate across calls in *acc (zero it first).
int dawn_debug_gemm_score_error(dawn_index *idx, const float *queries, size_t batch, dawn_score_error *acc) {
    int rc = check_alive(idx);
    if (rc) return rc;
    if (!queries || !acc || batch == 0) return fail(DAWN_ERR_INVALID, "null argument");
    if (idx->scalar == DAWN_SCALAR_I8) return fail(DAWN_ERR_INVALID, "fp16 / f32 storage only");
    std::shared_lock<std::shared_mutex> rd;
    size_t n = 0;
    float eps_scale = 1.0f;
    rc = snapshot_for_search(idx, rd, &n, &eps_scale);
    if (rc) return rc;
    if (n == 0 || n > 2048) return fail(DAWN_ERR_INVALID, "the index must hold 1..2048 rows (one candidate log per query)");
    WsLease lease(idx);
    SearchWs *ws = lease.ws;
    if (!ws) return fail(DAWN_ERR_CUDA, "cannot create a search workspace");
    rc = ensure_query_ws(idx, ws, batch, 1);
    if (rc) return rc;
    if ((rc = ensure_gemm_ws(idx, ws, gemm_workspace_bytes((int)batch)))) return rc;
    cudaStream_t s = ws->stream;
    memcpy(ws->h_queries, queries, batch * kDim * sizeof(float));
    CK(idx, cudaMemcpyAsync(ws->d_queries, ws->h_queries, batch * kDim * sizeof(float), cudaMemcpyHostToDevice, s));
    GemmSearch gs{};
    gs.corpus = idx->corpus;
    gs.labels = idx->labels;
    gs.n_rows = n;
    gs.queries = ws->d_queries;
    gs.n_queries = (int)batch;
    gs.kprime = 16;
    fill_gemm_knobs(idx, gs);
    gs.workspace = ws->d_gemm_ws;
    gs.final_lists = nullptr;
    gs.accum_slack = kGemmAccumSlack;
    gs.limit_score = -INFINITY;
    gs.debug_raw_scores = 1;
    const float *eps_q = nullptr;
    const uint2 *log = nullptr;
    const uint32_t *cnt = nullptr;
    const __half *q16 = nullptr;
    gs.eps_out = &eps_q;
    gs.debug_log_out = &log;
    gs.debug_cnt_out = &cnt;
    gs.debug_q16_out = &q16;
    CK(idx, launch_gemm_search(gs, s));
    unsigned long long *d_out = nullptr;
    CK(idx, cudaMalloc(&d_out, 48 * sizeof(unsigned long long)));
    CK(idx, cudaMemsetAsync(d_out, 0, 48 * sizeof(unsigned long long), s));
    CK(idx, launch_score_error(log, cnt, (int)batch, 2048, idx->corpus, ws->d_queries, q16, eps_q, d_out, s));
    unsigned long long h[48];
    CK(idx, cudaMemcpyAsync(h, d_out, sizeof h, cudaMemcpyDeviceToHost, s));
    CK(idx, cudaStreamSynchronize(s));
    cudaFree(d_out);
    auto as_double = [](unsigned long long u) { double d; memcpy(&d, &u, 8); return d; };
    auto upd = [](double &a, double b) { if (b > a) a = b; };
    upd(acc->max_mma_vs_f64, as_double(h[0]));
    upd(acc->max_seq_vs_f64, as_double(h[1]));
    upd(acc->max_mma_vs_seq, as_double(h[2]));
    upd(acc->max_err_over_eps_q, as_double(h[3]));
    acc->pairs += h[4];
    for (int b = 0; b < 40; b++) acc->hist[b] += h[8 + b];
    acc->scan_eps = kScanEps;
    acc->gemm_accum_slack = kGemmAccumSlack;
    acc->i8_dequant_slack = kI8DequantSlack;
    return DAWN_OK;
}

int dawn_index_set_option(dawn_index *idx, const char *key, int64_t value) {
    int rc = check_alive(idx);
    if (rc) return rc;
    if (!key) return fail(DAWN_ERR_INVALID, "key is null");
    if (!strcmp(key, "gemm_min_batch")) idx->gemm_min_batch = value;
    else if (!strcmp(key, "gemm_min_rows")) idx->gemm_min_rows = value;
    else if (!strcmp(key, "gemm_small_batch")) idx->gemm_small_batch = value;
    else if (!strcmp(key, "gemm_small_batch_rows")) idx->gemm_small_batch_rows = value;
    else if (!strcmp(key, "force_path")) idx->force_path = value;
    else if (!strcmp(key, "gemm_cta_group")) idx->gemm_cta_group = value;
    else if (!strcmp(key, "gemm_chunk_tiles")) idx->gemm_chunk_tiles = value;
    else if (!strcmp(key, "gemm_sequential_tiles")) idx->gemm_sequential_tiles = value;
    else if (!strcmp(key, "gemm_growth")) idx->gemm_growth = value;
    else if (!strcmp(key, "gemm_unit_sync")) idx->gemm_unit_sync = value;
    else if (!strcmp(key, "i8_tensor_min_batch")) idx->i8_tensor_min_batch = value;
    else if (!strcmp(key, "i8_tensor_chunk_rows")) idx->i8_tensor_chunk_rows = value < 65536 ? 65536 : value;
    else if (!strcmp(key, "i8_native")) idx->i8_native = value;
    else if (!strcmp(key, "shadow_i8")) idx->shadow_i8 = value;
    else if (!strcmp(key, "shadow_group_rows")) {
        if (value != 1 && value != 32) return fail(DAWN_ERR_INVALID, "shadow_group_rows must be 1 or 32, not %lld", (long long)value);
        std::lock_guard<std::mutex> lk(idx->mu);
        if (idx->shadow_group_rows != value) {  // the shadow is rebuilt with the new scales before the next search
            std::unique_lock<std::shared_mutex> wr(idx->corpus_mu);
            wait_device_searches(idx);
            drop_shadow(idx);
            idx->shadow_group_rows = value;
        }
    }
    else if (!strcmp(key, "shadow_single_rows")) idx->shadow_single_rows = value;
    else if (!strcmp(key, "shadow_big_k_rows")) idx->shadow_big_k_rows = value;
    else return fail(DAWN_ERR_INVALID, "unknown option '%s'", key);
    return DAWN_OK;
}

int dawn_index_set_profiling(dawn_index *idx, int enable) {
    int rc = check_alive(idx);
    if (rc) return rc;
    {
        std::lock_guard<std::mutex> lk(idx->dev_mu);
        drain_events(idx->dev_ws, idx->dev_ws->ws_used ? idx->dev_ws->ws_stream : idx->dev_ws->stream);
        merge_profile(idx, idx->dev_ws);
    }
    idx->profiling = enable != 0;
    return DAWN_OK;
}

int dawn_index_get_profile(dawn_index *idx, dawn_profile *out, int reset) {
    int rc = check_alive(idx);
    if (rc) return rc;
    if (!out) return fail(DAWN_ERR_INVALID, "out is null");
    {
        std::lock_guard<std::mutex> lk(idx->dev_mu);
        SearchWs *ws = idx->dev_ws;
        cudaStream_t s = ws->ws_used ? ws->ws_stream : ws->stream;
        drain_events(ws, s);
        merge_profile(idx, ws);
        // device-side counters (written by every finalize launch): wait for the device-API stream, then read
        if (ws->ws_used) CK(idx, cudaEventSynchronize(ws->ws_done));
        CK(idx, cudaMemcpy(idx->h_stats, idx->d_stats, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        if (reset) CK(idx, cudaMemset(idx->d_stats, 0, 4 * sizeof(uint32_t)));
    }
    std::lock_guard<std::mutex> lk(idx->prof_mu);
    *out = idx->prof;
    out->device_uncertified = idx->h_stats[0];
    out->device_status = idx->h_stats[1];
    {
        float e;
        memcpy(&e, &idx->h_stats[2], 4);
        out->max_selection_error = e;
    }
    if (reset) idx->prof = dawn_profile{};
    return DAWN_OK;
}

int dawn_merge_results_device(int device, const uint64_t *d_labels, const float *d_distances,
                              const uint32_t *d_counts, size_t n_lists, size_t list_stride_bytes,
                              size_t batch, size_t k, uint64_t *d_labels_out, float *d_distances_out,
                              uint32_t *d_counts_out, void *stream) {
    if (!d_labels || !d_distances || !d_counts || !d_labels_out || !d_distances_out || !d_counts_out)
        return fail(DAWN_ERR_INVALID, "null device pointer");
    if (k == 0 || k > DAWN_MAX_K || n_lists == 0 || n_lists * k > 1024)
        return fail(DAWN_ERR_INVALID, "merge shape out of range (n_lists=%zu k=%zu; n_lists*k must be <= 1024)",
                    n_lists, k);
    if (batch == 0) return DAWN_OK;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess)
        e = launch_merge_results(d_labels, d_distances, d_counts, (int)n_lists, list_stride_bytes, (int)batch, (int)k,
                                 d_labels_out, d_distances_out, d_counts_out, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail(DAWN_ERR_CUDA, "merge launch failed: %s", cudaGetErrorString(e));
    return DAWN_OK;
}

}  // extern "C"

// ------------------------------------------------------------------ small kernels

namespace {

// K7 (device side of the sharded search): merge n_lists sorted result lists per query.
// Order: distance ascending, label ascending, then list index (strict).  One CTA per query,
// one thread per input entry; rank = position in own list + binary-searched counts in the others.
// A label that an EARLIER list already holds at the same distance is the same page stored on two
// shards; it is dropped, like BestResults::insert drops an id it already contains
// (/root/reference/src/search/best_results.rs:46,57).
__global__ void __launch_bounds__(1024) merge_results_kernel(
    const uint64_t *__restrict__ labels, const float *__restrict__ dist, const uint32_t *__restrict__ counts,
    int n_lists, size_t stride_l, size_t stride_d, size_t stride_c, int batch, int k,
    uint64_t *__restrict__ labels_out, float *__restrict__ dist_out, uint32_t *__restrict__ counts_out) {
    __shared__ uint64_t s_lab[1024];
    __shared__ float s_dist[1024];
    __shared__ uint64_t s_lab2[1024];
    __shared__ float s_dist2[1024];
    __shared__ uint8_t s_dup[1024];
    __shared__ int s_cnt[64], s_cnt2[64];
    const int qi = blockIdx.x;
    const int tid = threadIdx.x;
    const int total = n_lists * k;
    // list l's arrays start l * stride bytes after the base pointers (dense arrays or one packed
    // block per shard as it arrives from the all-gather)
    if (tid < n_lists)
        s_cnt[tid] = min((int)reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(counts) + tid * stride_c)[qi], k);
    if (tid < total) {
        const int l = tid / k, p = tid % k;
        s_lab[tid] = reinterpret_cast<const uint64_t *>(reinterpret_cast<const char *>(labels) + l * stride_l)[(size_t)qi * k + p];
        s_dist[tid] = reinterpret_cast<const float *>(reinterpret_cast<const char *>(dist) + l * stride_d)[(size_t)qi * k + p];
    }
    __syncthreads();
    // ---- cross-shard duplicates: (distance, label) found in a list with a smaller index
    bool dup = false;
    if (tid < total) {
        const int l = tid / k, p = tid % k;
        if (p < s_cnt[l]) {
            const float d = s_dist[tid];
            const uint64_t lab = s_lab[tid];
            for (int o = 0; o < l && !dup; o++) {
                int lo = 0, hi = s_cnt[o];
                while (lo < hi) {  // first entry of list o that is not before (d, lab)
                    const int mid = (lo + hi) >> 1;
                    const float od = s_dist[o * k + mid];
                    const uint64_t ol = s_lab[o * k + mid];
                    if (od < d || (od == d && ol < lab)) lo = mid + 1;
                    else hi = mid;
                }
                dup = lo < s_cnt[o] && s_dist[o * k + lo] == d && s_lab[o * k + lo] == lab;
            }
        }
        s_dup[tid] = dup ? 1 : 0;
    }
    const uint64_t *L = s_lab;
    const float *D = s_dist;
    const int *C = s_cnt;
    if (__syncthreads_or(dup ? 1 : 0)) {  // rare: compact every list without its duplicates
        if (tid < total) {
            const int l = tid / k, p = tid % k;
            if (p < s_cnt[l] && !dup) {
                int before = 0;
                for (int j = 0; j < p; j++) before += s_dup[l * k + j];
                s_lab2[l * k + p - before] = s_lab[tid];
                s_dist2[l * k + p - before] = s_dist[tid];
            }
        }
        if (tid < n_lists) {
            int dups = 0;
            for (int j = 0; j < s_cnt[tid]; j++) dups += s_dup[tid * k + j];
            s_cnt2[tid] = s_cnt[tid] - dups;
        }
        __syncthreads();
        L = s_lab2;
        D = s_dist2;
        C = s_cnt2;
    }
    int all = 0;
    for (int l = 0; l < n_lists; l++) all += C[l];
    if (tid < total) {
        const int l = tid / k, p = tid % k;
        if (p < C[l]) {
            const float d = D[tid];
            const uint64_t lab = L[tid];
            int rank = p;
            for (int o = 0; o < n_lists; o++) {
                if (o == l) continue;
                int lo = 0, hi = C[o];
                while (lo < hi) {  // count entries of list o that come before (d, lab, l)
                    const int mid = (lo + hi) >> 1;
                    const float od = D[o * k + mid];
                    const uint64_t ol = L[o * k + mid];
                    const bool before = od < d || (od == d && (ol < lab || (ol == lab && o < l)));
                    if (before) lo = mid + 1;
                    else hi = mid;
                }
                rank += lo;
            }
            if (rank < k) {
                labels_out[(size_t)qi * k + rank] = lab;
                dist_out[(size_t)qi * k + rank] = d;
            }
        }
    }
    if (tid == 0) counts_out[qi] = (uint32_t)min(all, k);
}

__global__ void __launch_bounds__(256) find_label_kernel(const uint64_t *__restrict__ labels, size_t n,
                                                         uint64_t label, uint32_t *__restrict__ row_out) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        if (labels[i] == label) atomicMin(row_out, (uint32_t)i);
}

// Norm gate over stored rows, one warp per row (vector.rs:181-192 applied to what is actually stored).  stats[3] counts the odd
// rows: an fp16 row with an inf / NaN component or one at +-65504 (the saturated copy of an f32 value out of the fp16 range),
// an int8 row with an infinite scale.  An int8 row whose squared norm overflows f32 (components ~1e30) still gets its finite
// norm, so the eps scale covers it.
__global__ void __launch_bounds__(256) verify_rows_kernel(const uint8_t *__restrict__ arena, int scalar, size_t first, size_t n,
                                                          uint32_t *__restrict__ stats) {
    const int lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    uint32_t bad = 0, odd_rows = 0;
    float vmax = 0.f, vmin = __int_as_float(0x7f800000);
    for (size_t r = warp; r < n; r += n_warps) {
        const size_t row = first + r;
        float acc = 0.f, isf = 0.f, sc = 1.f;
        bool odd = false;
        if (scalar == 0) {
            const __half *src = reinterpret_cast<const __half *>(arena) + row * kDim;
            const uint4 u = *reinterpret_cast<const uint4 *>(src + lane * 8);
            const uint2 v = *reinterpret_cast<const uint2 *>(src + 256 + lane * 4);
            const __half2 *h = reinterpret_cast<const __half2 *>(&u);
            const __half2 *g = reinterpret_cast<const __half2 *>(&v);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const float2 x = __half22float2(h[j]);
                acc = fmaf(x.x, x.x, acc);
                acc = fmaf(x.y, x.y, acc);
                odd |= !(fabsf(x.x) < 65504.f) || !(fabsf(x.y) < 65504.f);
            }
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const float2 x = __half22float2(g[j]);
                acc = fmaf(x.x, x.x, acc);
                acc = fmaf(x.y, x.y, acc);
                odd |= !(fabsf(x.x) < 65504.f) || !(fabsf(x.y) < 65504.f);
            }
        } else {
            const int8_t *src = reinterpret_cast<const int8_t *>(arena + i8_row_offset(row));
            sc = *reinterpret_cast<const float *>(arena + i8_scale_offset(row));
            odd = !(sc < INFINITY);
            const uint2 u = *reinterpret_cast<const uint2 *>(src + lane * 8);
            const uint32_t v = *reinterpret_cast<const uint32_t *>(src + 256 + lane * 4);
            const int8_t *a = reinterpret_cast<const int8_t *>(&u);
            const int8_t *b = reinterpret_cast<const int8_t *>(&v);
            int isum = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) isum += (int)a[j] * (int)a[j];
#pragma unroll
            for (int j = 0; j < 4; j++) isum += (int)b[j] * (int)b[j];
            acc = (float)isum * sc * sc;
            isf = (float)isum;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            acc += __shfl_xor_sync(0xffffffffu, acc, off);
            isf += __shfl_xor_sync(0xffffffffu, isf, off);
        }
        odd = __any_sync(0xffffffffu, odd);
        float len = sqrtf(acc);
        if (!(len < INFINITY) && !odd) len = sqrtf(isf) * sc;  // int8 only: isum * sc * sc overflowed
        const bool finite = len == len && len < __int_as_float(0x7f800000);
        if (!(finite && len > 0.99f && len < 1.01f)) bad++;
        if (odd) odd_rows++;
        if (finite) {
            vmax = fmaxf(vmax, len);
            vmin = fminf(vmin, len);
        }
    }
    if (lane == 0) {
        if (bad) atomicAdd(&stats[0], bad);
        if (odd_rows) atomicAdd(&stats[3], odd_rows);
        atomicMax(&stats[1], __float_as_uint(vmax));      // norms are >= 0: the bit pattern orders like the value
        atomicMax(&stats[2], ~__float_as_uint(vmin));     // min kept inverted so that zero-initialised memory means "none yet"
    }
}

__global__ void __launch_bounds__(256) iota_labels_kernel(uint64_t *__restrict__ dst, uint64_t first, size_t n) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = first + i;
}

cudaError_t launch_merge_results(const uint64_t *labels, const float *dist, const uint32_t *counts, int n_lists,
                                 size_t list_stride_bytes, int batch, int k, uint64_t *labels_out, float *dist_out,
                                 uint32_t *counts_out, cudaStream_t s) {
    if (n_lists > 64) return cudaErrorInvalidValue;
    size_t sl = list_stride_bytes, sd = list_stride_bytes, sc = list_stride_bytes;
    if (list_stride_bytes == 0) {  // dense [n_lists][batch][k] arrays
        sl = (size_t)batch * k * sizeof(uint64_t);
        sd = (size_t)batch * k * sizeof(float);
        sc = (size_t)batch * sizeof(uint32_t);
    }
    merge_results_kernel<<<batch, 1024, 0, s>>>(labels, dist, counts, n_lists, sl, sd, sc, batch, k, labels_out,
                                                dist_out, counts_out);
    return cudaGetLastError();
}

cudaError_t launch_find_label(const uint64_t *labels, size_t n, uint64_t label, uint32_t *row_out,
                              cudaStream_t s) {
    cudaError_t e = cudaMemsetAsync(row_out, 0xFF, sizeof(uint32_t), s);
    if (e != cudaSuccess) return e;
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    find_label_kernel<<<(unsigned)blocks, 256, 0, s>>>(labels, n, label, row_out);
    return cudaGetLastError();
}

cudaError_t launch_verify_rows(const void *arena, int scalar, size_t first, size_t n, uint32_t *stats, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    size_t blocks = (n + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    verify_rows_kernel<<<(unsigned)blocks, 256, 0, s>>>(static_cast<const uint8_t *>(arena), scalar, first, n, stats);
    return cudaGetLastError();
}

}  // namespace

namespace dawn {
// int8 shadow of fp16 rows: x8 = rint(x16 / s), written in the blocked int8 layout the int8 kernels read (8 rows x 384 B +
// 8 f32 scales per 3104-byte block).  With group_rows = 32 every row of a group of 32 rows (aligned to the absolute row
// index) gets the group's scale s = max absmax / 127: a group is exactly one 32-column chunk of gemm_i8_topk_kernel's
// epilogue, whose first filter level multiplies the chunk's largest HI by its largest scale, so with one scale per chunk that
// test is as tight as the per-element test.  Per-row scales (group_rows = 1) spread from 0.87x to 1.17x of the median and
// make that level 12-20x looser (tools/shadow_filter_model.py).  The price is a coarser step for the rows of a group with a
// smaller absmax: ~8-10 % more filter survivors.
// Only rows [first, first + n) are written and only they enter their group's maximum: rows below `first` may already be read
// by searches in flight, so a group that straddles an append keeps its old rows' scale and its new rows get their own.
// The chunk test takes the largest scale of the chunk, so such a chunk stays rigorous, only looser.
// Zero rows and rows with inf / NaN are stored as zeros under the group's scale and are left out of its maximum; a group of
// nothing but such rows gets scale 1.  Such a row can be a hit (an inf component scores +-inf), so the searches do not use the
// shadow while the norm gate counts one (search_enqueue).
// One block of 8 warps per group, 4 rows per warp.  kappa_bits collects max ||x16 / s - x8|| over the rows with the stored s
// (<= sqrt(384) / 2 = 9.8 for any s >= absmax / 127, ~5.7-6.3 on real rows): the filter's rigorous bound on a row's own
// quantisation error is ||q|| * kappa * s_row.
constexpr int kShadowGroupRows = 32;
__global__ void __launch_bounds__(256) shadow_quantize_kernel(const __half *__restrict__ corpus, uint8_t *__restrict__ arena,
                                                              size_t first, size_t n, int group_rows,
                                                              uint32_t *__restrict__ kappa_bits) {
    __shared__ float s_amax[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t end = first + n;
    const size_t g_end = (end + kShadowGroupRows - 1) / kShadowGroupRows;
    float kmax = 0.f;
    for (size_t g = first / kShadowGroupRows + blockIdx.x; g < g_end; g += gridDim.x) {
        float amax[4], wmax = 0.f;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const size_t row = g * kShadowGroupRows + warp + 8 * i;
            float m = 0.f;
            if (row >= first && row < end) {
                const uint2 *src = reinterpret_cast<const uint2 *>(corpus + row * kDim) + lane * 3;  // 12 halfs per lane
#pragma unroll
                for (int j = 0; j < 3; j++) {
                    const uint2 u = __ldg(src + j);
                    const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&u.x));
                    const float2 b = __half22float2(*reinterpret_cast<const __half2 *>(&u.y));
                    m = fmaxf(fmaxf(m, fmaxf(fabsf(a.x), fabsf(a.y))), fmaxf(fabsf(b.x), fabsf(b.y)));
                }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
            if (!(m < INFINITY)) m = 0.f;
            amax[i] = m;
            wmax = fmaxf(wmax, m);
        }
        if (group_rows > 1) {
            if (lane == 0) s_amax[warp] = wmax;
            __syncthreads();
            wmax = s_amax[0];
#pragma unroll
            for (int w = 1; w < 8; w++) wmax = fmaxf(wmax, s_amax[w]);
            __syncthreads();  // s_amax is rewritten for the next group
        }
        // second pass over the same rows (L1 / L2 hits): keeping all four in registers through the divisions spills
#pragma unroll 1
        for (int i = 0; i < 4; i++) {
            const size_t row = g * kShadowGroupRows + warp + 8 * i;
            if (row < first || row >= end) continue;
            const float ra = i == 0 ? amax[0] : i == 1 ? amax[1] : i == 2 ? amax[2] : amax[3];
            const float m = group_rows > 1 ? wmax : ra;
            const float sc = m > 0.f ? __fdiv_rn(m, 127.0f) : 1.0f;
            const uint2 *src = reinterpret_cast<const uint2 *>(corpus + row * kDim) + lane * 3;
            uint32_t packed[3];
            float err2 = 0.f;
#pragma unroll
            for (int j = 0; j < 3; j++) {
                const uint2 u = __ldg(src + j);
                const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&u.x));
                const float2 b = __half22float2(*reinterpret_cast<const __half2 *>(&u.y));
                const float xs[4] = {a.x, a.y, b.x, b.y};
                uint32_t w = 0;
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const float v = ra > 0.f ? xs[e] : 0.f;
                    const float t = __fdiv_rn(v, sc);
                    const int qv = max(-127, min(127, (int)rintf(t)));
                    const float d = t - (float)qv;
                    err2 = fmaf(d, d, err2);
                    w |= ((uint32_t)(qv & 0xff)) << (8 * e);
                }
                packed[j] = w;
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) err2 += __shfl_xor_sync(0xffffffffu, err2, off);
            uint32_t *dst = reinterpret_cast<uint32_t *>(arena + i8_row_offset((uint32_t)row)) + lane * 3;
            dst[0] = packed[0], dst[1] = packed[1], dst[2] = packed[2];
            if (lane == 0) *reinterpret_cast<float *>(arena + i8_scale_offset((uint32_t)row)) = sc;
            kmax = fmaxf(kmax, sqrtf(err2) * 1.00001f);
        }
    }
    if (lane == 0 && kmax > 0.f) atomicMax(kappa_bits, __float_as_uint(kmax));
}

cudaError_t launch_shadow_quantize(const __half *corpus, uint8_t *arena, size_t first, size_t n, int group_rows,
                                   uint32_t *kappa_bits, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    if (group_rows != 1 && group_rows != kShadowGroupRows) return cudaErrorInvalidValue;
    const size_t groups = (first + n + kShadowGroupRows - 1) / kShadowGroupRows - first / kShadowGroupRows;
    size_t blocks = groups;
    if (blocks > 148 * 8) blocks = 148 * 8;
    shadow_quantize_kernel<<<(unsigned)blocks, 256, 0, s>>>(corpus, arena, first, n, group_rows, kappa_bits);
    return cudaGetLastError();
}

// distance_limit on the device API: results ascend, so "drop distance >= limit" is a cut of the count
__global__ void truncate_by_limit_kernel(const float *__restrict__ dist, uint32_t *__restrict__ counts, int batch, int k,
                                         float limit) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    const uint32_t c = counts[b];
    uint32_t keep = 0;
    while (keep < c && dist[(size_t)b * k + keep] < limit) keep++;
    counts[b] = keep;
}

cudaError_t launch_truncate_by_limit(const float *dist, uint32_t *counts, size_t batch, size_t k, float limit, cudaStream_t s) {
    truncate_by_limit_kernel<<<(unsigned)((batch + 127) / 128), 128, 0, s>>>(dist, counts, (int)batch, (int)k, limit);
    return cudaGetLastError();
}

cudaError_t launch_iota_labels(uint64_t *dst, uint64_t first, size_t n, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    iota_labels_kernel<<<(unsigned)blocks, 256, 0, s>>>(dst, first, n);
    return cudaGetLastError();
}
}  // namespace dawn
