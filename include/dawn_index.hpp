// dawn_index.hpp -- header-only C++17 host mirror of the reference's interfaces for the vector
// top-k hot path, layered on the C ABI in dawn_index.h.  The reference is compiled code (Rust) and
// there is no Rust toolchain in this build image, so this is the compiled-language host side; the
// Rust shim with the same shape is in rust/src/index/gpu_index.rs (INTEGRATION.md).
//
//   dawn::ffi::{IndexOptions, MetricKind, ScalarKind, Matches, Index, new_index, Batcher}
//        == usearch::ffi as used at /root/reference/src/search/search_provider.rs:32-42,102,115-117,
//           133,149,178,214,221,246,280-284 (same method names, argument meaning; C++ exceptions
//           where the cxx bridge returned Result::Err)
//   dawn::{EM_LEN, is_normalized, normalize, vector_length, distance_cosine}
//        == src/search/vector.rs:26,128-134,181-197
//   dawn::BestResults<T>
//        == src/search/best_results.rs:22-108 (kept as is, including arrival-order ties and the
//           worst_distance()==0-until-full quirk; the device merge uses a total order instead)
//   dawn::SearchProvider
//        == src/search/search_provider.rs:44-333 with the SQLite row store replaced by an in-memory
//           map (SQLite is outside the hot path): new / search_embedding (k = 20) / search_like /
//           embedding_for_page / insert (1M cap, URL dedupe, norm gate, reserve +1024) / save /
//           shutdown / stats
#pragma once

#include <cmath>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "dawn_index.h"

namespace dawn {

constexpr std::size_t EM_LEN = DAWN_DIMENSIONS;  // src/search/vector.rs:26

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

inline void check(int rc) {
    if (rc != DAWN_OK) throw Error(rc, dawn_last_error());
}

// ---- src/search/vector.rs --------------------------------------------------------------------
inline float vector_length(const float *v) { return dawn_vector_length(v); }   // :181-183
inline bool is_normalized(const float *v) { return dawn_is_normalized(v) != 0; }  // :185-192
inline void normalize(std::vector<float> &v) { dawn_normalize(v.data()); }      // :194-197
inline std::vector<std::uint8_t> to24(const std::vector<float> &v) {               // :74-86
    if (v.size() != EM_LEN) throw Error(DAWN_ERR_INVALID, "embedding must have 384 dimensions");
    std::vector<std::uint8_t> out(3 * EM_LEN);
    dawn_encode_i24(v.data(), out.data());
    return out;
}
inline std::vector<float> from24(const std::vector<std::uint8_t> &data) {          // :52-72 (ensure!s the norm)
    if (data.size() != 3 * EM_LEN) throw Error(DAWN_ERR_INVALID, "i24 embedding must be 1152 bytes");
    std::vector<float> v(EM_LEN);
    if (dawn_decode_i24(data.data(), v.data()) != DAWN_OK) throw Error(DAWN_ERR_INVALID, "Embedding is not normalized");
    return v;
}
inline float distance_cosine(const float *a, const float *b) {                   // :128-134
    float result = 0.0f;
    for (std::size_t i = 0; i < EM_LEN; i++) result += a[i] * b[i];
    return 1.0f - result;
}

// ---- src/search/best_results.rs ----------------------------------------------------------------
template <class T>
struct NodeReference {  // :22-26
    std::size_t id;
    T distance;
};

template <class T>
class BestResults {  // :28-108
    std::vector<NodeReference<T>> results_;
    std::size_t worst_result_index_ = 0;
    T worst_distance_ = T(0);
    std::size_t size_;

    bool contains_id(std::size_t id) const {
        for (auto &x : results_)
            if (x.id == id) return true;
        return false;
    }
    void update_worst() {
        worst_result_index_ = 0;
        worst_distance_ = results_[0].distance;
        for (std::size_t i = 1; i < results_.size(); i++)
            if (results_[i].distance > worst_distance_) {
                worst_distance_ = results_[i].distance;
                worst_result_index_ = i;
            }
    }

public:
    explicit BestResults(std::size_t size) : size_(size) { results_.reserve(size); }
    bool insert(NodeReference<T> r) {  // :44-65
        if (results_.size() < size_) {
            if (contains_id(r.id)) return false;
            results_.push_back(r);
            if (results_.size() == size_) update_worst();
            return true;
        }
        if (r.distance < worst_distance_) {
            if (contains_id(r.id)) return false;
            results_[worst_result_index_] = r;
            update_worst();
            return true;
        }
        return false;
    }
    void sort() {  // :71-79 (stable, ascending distance)
        if (results_.empty()) return;
        for (std::size_t i = 1; i < results_.size(); i++) {
            auto x = results_[i];
            std::size_t j = i;
            while (j > 0 && results_[j - 1].distance > x.distance) {
                results_[j] = results_[j - 1];
                j--;
            }
            results_[j] = x;
        }
        worst_result_index_ = results_.size() - 1;
        worst_distance_ = results_.back().distance;
    }
    const std::vector<NodeReference<T>> &results() const { return results_; }
    std::size_t len() const { return results_.size(); }
    void clear() { results_.clear(); }
    T worst_distance() const { return worst_distance_; }
};

// ---- usearch::ffi -------------------------------------------------------------------------------
namespace ffi {

enum class MetricKind { IP };
enum class ScalarKind { F32, F16, F8 };  // F32 is accepted and stored as F16 on the device; F8 -> int8 storage

struct IndexOptions {  // search_provider.rs:35-42
    std::size_t dimensions = EM_LEN;
    MetricKind metric = MetricKind::IP;
    ScalarKind quantization = ScalarKind::F32;
    std::size_t connectivity = 0;      // meaningless for an exact scan, accepted for source compatibility
    std::size_t expansion_add = 0;
    std::size_t expansion_search = 0;
    int device = 0;                    // addition: CUDA device ordinal
};

struct Matches {  // search_provider.rs:221
    std::vector<std::uint64_t> labels;
    std::vector<float> distances;
};

class Index {
    dawn_index *h_ = nullptr;

public:
    explicit Index(const IndexOptions &o) {
        dawn_options opts{};
        opts.dimensions = static_cast<std::uint32_t>(o.dimensions);
        opts.metric = DAWN_METRIC_IP;
        opts.scalar = o.quantization == ScalarKind::F8 ? DAWN_SCALAR_I8 : DAWN_SCALAR_F16;
        opts.device = o.device;
        check(dawn_index_create(&opts, &h_));
    }
    ~Index() { dawn_index_free(h_); }
    Index(const Index &) = delete;
    Index &operator=(const Index &) = delete;

    void reserve(std::size_t capacity) const { check(dawn_index_reserve(h_, capacity)); }         // :133,282
    void add(std::uint64_t label, const std::vector<float> &v) const {                            // :149,284
        if (v.size() != EM_LEN) throw Error(DAWN_ERR_INVALID, "vector must have 384 dimensions");
        check(dawn_index_add(h_, label, v.data()));
    }
    void add_batch(const std::vector<std::uint64_t> &labels, const std::vector<float> &vectors) const {
        if (vectors.size() != labels.size() * EM_LEN) throw Error(DAWN_ERR_INVALID, "vectors must be labels x 384");
        check(dawn_index_add_batch(h_, labels.data(), vectors.data(), labels.size()));
    }
    // Drop every stored vector with this label / these labels; returns the vectors removed.  Update = remove + add.
    std::size_t remove(std::uint64_t label) const {
        std::size_t n = 0;
        check(dawn_index_remove(h_, label, &n));
        return n;
    }
    std::size_t remove_batch(const std::vector<std::uint64_t> &labels) const {
        std::size_t n = 0;
        check(dawn_index_remove_batch(h_, labels.data(), labels.size(), &n));
        return n;
    }
    Matches search(const std::vector<float> &query, std::size_t count) const {                    // :214
        if (query.size() != EM_LEN) throw Error(DAWN_ERR_INVALID, "query must have 384 dimensions");
        Matches m;
        m.labels.resize(count);
        m.distances.resize(count);
        std::size_t n = 0;
        check(dawn_index_search(h_, query.data(), count, m.labels.data(), m.distances.data(), &n));
        m.labels.resize(n);
        m.distances.resize(n);
        return m;
    }
    std::size_t size() const { return dawn_index_size(h_); }            // :246,280
    std::size_t capacity() const { return dawn_index_capacity(h_); }    // :280
    std::size_t dimensions() const { return dawn_index_dimensions(h_); }
    void save(const std::string &path) const { check(dawn_index_save(h_, path.c_str())); }  // :117,178
    void load(const std::string &path) const { check(dawn_index_load(h_, path.c_str())); }  // :115
    void view(const std::string &path) const { load(path); }  // examples_old/search_usearch.rs:47
    std::vector<float> get(std::uint64_t label) const {
        std::vector<float> v(EM_LEN);
        check(dawn_index_get(h_, label, v.data()));
        return v;
    }
    // ---- the callers and formats either side of the path (SURVEY 8f) --------------------------------
    // UdpPacket::Search{distance_limit} (src/net/udp_packets.rs:29-39): hits with distance >= limit are dropped
    // (src/net/udp_service.rs:196-199); the limit is pushed down into the scan kernels.
    Matches search_limit(const std::vector<float> &query, std::size_t count, float distance_limit) const {
        if (query.size() != EM_LEN) throw Error(DAWN_ERR_INVALID, "query must have 384 dimensions");
        Matches m;
        m.labels.resize(count);
        m.distances.resize(count);
        std::size_t n = 0;
        check(dawn_index_search_limit(h_, query.data(), count, distance_limit, m.labels.data(), m.distances.data(), &n));
        m.labels.resize(n);
        m.distances.resize(n);
        return m;
    }
    // The peer side of a remote search: the 1152-byte i24 embedding straight off the wire (vector.rs:48-87).
    Matches search_i24(const std::vector<std::uint8_t> &wire, std::size_t count, bool has_limit = false,
                       float distance_limit = 0.0f) const {
        if (wire.size() != 3 * EM_LEN) throw Error(DAWN_ERR_INVALID, "i24 embedding must be 1152 bytes");
        Matches m;
        m.labels.resize(count);
        m.distances.resize(count);
        std::size_t n = 0;
        check(dawn_index_search_i24(h_, wire.data(), count, has_limit ? 1 : 0, distance_limit, m.labels.data(),
                                    m.distances.data(), &n));
        m.labels.resize(n);
        m.distances.resize(n);
        return m;
    }
    std::vector<std::uint8_t> get_i24(std::uint64_t label) const {  // GetEmbedding over UDP (udp_service.rs:254-276)
        std::vector<std::uint8_t> v(3 * EM_LEN);
        check(dawn_index_get_i24(h_, label, v.data()));
        return v;
    }
    // SearchProvider::verify over the device corpus (search_provider.rs:289-327): rows failing the norm gate, min / max norm.
    struct VerifyResult { std::size_t bad_rows; float min_norm, max_norm; };
    VerifyResult verify() const {
        VerifyResult r{0, 0.f, 0.f};
        check(dawn_index_verify(h_, &r.bad_rows, &r.min_norm, &r.max_norm));
        return r;
    }
    // Tuning knobs (dawn_index.h).  set_option("shadow_i8", 1): the fp16 corpus also keeps an int8 copy of itself that is only
    // used to FILTER on the int8 tensor cores; candidates are re-scored on the fp16 rows, results do not change.
    void set_option(const std::string &key, std::int64_t value) const { check(dawn_index_set_option(h_, key.c_str(), value)); }
    dawn_index *handle() const { return h_; }
};

// Micro-batching front for SearchService (src/search/search_service.rs:55-104): many threads call search() with one
// query each and are answered in batches (what arrived while the previous batch was on the GPU; a lone caller never waits).
// Must not outlive the index.
class Batcher {
    dawn_batcher *b_ = nullptr;

public:
    Batcher(const Index &index, std::size_t max_batch, std::uint32_t max_wait_us) {
        check(dawn_batcher_create(index.handle(), max_batch, max_wait_us, &b_));
    }
    ~Batcher() { dawn_batcher_free(b_); }
    Batcher(const Batcher &) = delete;
    Batcher &operator=(const Batcher &) = delete;
    Matches search(const std::vector<float> &query, std::size_t count) const {
        if (query.size() != EM_LEN) throw Error(DAWN_ERR_INVALID, "query must have 384 dimensions");
        Matches m;
        m.labels.resize(count);
        m.distances.resize(count);
        std::size_t n = 0;
        if (dawn_batcher_search(b_, query.data(), count, m.labels.data(), m.distances.data(), &n) != DAWN_OK)
            throw Error(DAWN_ERR_INTERNAL, dawn_batcher_last_error());
        m.labels.resize(n);
        m.distances.resize(n);
        return m;
    }
};

inline std::unique_ptr<Index> new_index(const IndexOptions &o) { return std::make_unique<Index>(o); }  // :102

}  // namespace ffi

// ---- src/search/search_provider.rs ------------------------------------------------------------
struct ExtractedPage {  // src/search/page_source.rs
    std::string url, title, text;
};

struct FoundPage {  // search_provider.rs:51-59
    std::string instance_id;
    std::size_t page_id;
    float distance;
    std::string url, title, text;
};

struct SearchResult {  // :44-49
    std::vector<FoundPage> pages;
    std::size_t servers_contacted = 0;
    std::size_t pages_searched = 0;
};

struct SearchStats {  // :61-64
    std::size_t pages_indexed;
};

class SearchProvider {  // :66-73
    std::unique_ptr<ffi::Index> index_;
    struct Row {
        std::string url, title, text;
    };
    std::unordered_map<std::uint64_t, Row> rows_;                 // stands in for the SQLite `page` table (:85-91)
    std::unordered_map<std::string, std::uint64_t> find_by_url_;  // CREATE INDEX find_by_url (:93-98)
    std::uint64_t last_rowid_ = 0;
    std::string data_dir_;

public:
    static constexpr std::size_t kSearchCount = 20;     // :214
    static constexpr std::size_t kMaxPages = 1000000;   // :164-166

    explicit SearchProvider(std::string data_dir, int device = 0) : data_dir_(std::move(data_dir)) {  // :76-125
        ffi::IndexOptions o;  // INDEX_OPTIONS :35-42
        o.device = device;
        index_ = ffi::new_index(o);
    }

    bool local_space_available() const { return rows_.size() < kMaxPages; }  // :164-166

    SearchResult search_embedding(const std::vector<float> &query_embedding) const {  // :202-248
        if (query_embedding.size() != EM_LEN || !is_normalized(query_embedding.data()))
            throw Error(DAWN_ERR_INVALID, "Search vector is not normalized");
        SearchResult r;
        ffi::Matches results = index_->search(query_embedding, kSearchCount);
        for (std::size_t i = 0; i < results.labels.size(); i++) {
            auto it = rows_.find(results.labels[i]);
            if (it == rows_.end()) continue;  // "Page not found in DB"
            r.pages.push_back(FoundPage{std::string(), static_cast<std::size_t>(results.labels[i]), results.distances[i],
                                        it->second.url, it->second.title, it->second.text});
        }
        r.servers_contacted = 0;
        r.pages_searched = index_->size();
        return r;
    }

    std::vector<float> embedding_for_page(std::size_t id) const {  // :183-195 (served from the device corpus)
        if (!rows_.count(id)) throw Error(DAWN_ERR_INVALID, "Page not found in DB: " + std::to_string(id));
        return index_->get(id);
    }

    SearchResult search_like(std::size_t id) const { return search_embedding(embedding_for_page(id)); }  // :197-200

    void insert(const ExtractedPage &page, const std::vector<float> &q) {  // :250-286
        if (!local_space_available()) throw Error(DAWN_ERR_CAPACITY, "No space available");
        if (find_by_url_.count(page.url)) return;  // "Already have with id"
        if (q.size() != EM_LEN || !is_normalized(q.data())) throw Error(DAWN_ERR_INVALID, "Insert embedding is not normalized");
        const std::uint64_t id = ++last_rowid_;  // last_insert_rowid()
        rows_[id] = Row{page.url, page.title, page.text};
        find_by_url_[page.url] = id;
        if (index_->size() == index_->capacity()) index_->reserve(index_->size() + 1024);  // :280-283
        index_->add(id, q);
    }

    void save() const { index_->save(data_dir_ + "/index.dawn"); }  // :168-181
    void shutdown() const { save(); }                               // :155-158
    SearchStats stats() const { return SearchStats{rows_.size()}; }  // :329-332
};

}  // namespace dawn
