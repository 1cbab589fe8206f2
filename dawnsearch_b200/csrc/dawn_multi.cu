// dawn_multi.cu -- the multi-GPU layer for a SINGLE-PROCESS caller (the reference binary is one
// process, /root/reference/src/bin/dawnsearch.rs:59-128): the corpus is sharded over the GPUs of one
// box, every GPU answers the batch from its shard, then ONE NCCL all-gather over NVLink / NVSwitch
// moves every shard's packed block of k (label, distance) pairs per query to every GPU
// (ncclCommInitAll over the listed devices, one communicator per shard, the collective issued as one
// group) and merge_results_kernel merges them on the first device -- the shape of the reference's
// scatter / gather / merge across WAN peers (src/net/udp_service.rs:314-330,
// src/search/search_service.rs:201-277).  Exchange "peer" (one cudaMemcpyPeerAsync per shard into the
// first device's memory) is kept for handles that list one device twice (tests on a one-GPU box), where
// NCCL cannot form a communicator, and as the A/B partner of the collective
// (dawn_multi_set_option "exchange").
// (The one-process-per-GPU variant of the same exchange under torch.distributed is dawnsearch_b200/sharded.py.)
//
// Exactness: shards return bit-exact distances, the merge orders by (distance, label), so the
// answer equals a single index holding everything as long as every label is stored once (a label
// stored on two shards at the same distance comes back once: include/dawn_index.h,
// dawn_merge_results_device).  Queries a shard could not certify are re-run on that shard through
// the exact scan before the merge.
#include <atomic>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <cmath>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types and prototypes only: the library is bound at run time, see NcclApi

#include "../../include/dawn_index.h"

namespace {

thread_local std::string g_multi_err;

// NCCL is bound at RUN time (dlopen) instead of through a DT_NEEDED entry, for two reasons:
//  * a process that already holds an NCCL must keep using THAT one.  The test / bench harness imports torch, whose
//    libtorch_cuda.so needs its own bundled libnccl.so.2 (2.28, with symbols the system 2.27 lacks); the dynamic loader
//    matches by SONAME, so whichever libnccl.so.2 is mapped first serves everybody -- a DT_NEEDED on the system copy made
//    `import torch` fail with "undefined symbol: ncclDevCommCreate" whenever libdawn_b200.so happened to be loaded first;
//  * single-GPU users of the library need no NCCL at all.
// Resolution order: an NCCL already mapped into the process, then $DAWN_NCCL_LIB, then "libnccl.so.2" by name.
struct NcclApi {
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int *) = nullptr;
    std::string origin;
    bool ok = false;
};

const NcclApi &nccl_api() {
    static NcclApi api = [] {
        NcclApi a;
        void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        a.origin = "already loaded in the process";
        if (!h) {
            if (const char *env = getenv("DAWN_NCCL_LIB")) {
                h = dlopen(env, RTLD_NOW | RTLD_LOCAL);
                a.origin = env;
            }
        }
        if (!h) {
            h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
            a.origin = "libnccl.so.2";
        }
        if (!h) {
            a.origin = std::string("libnccl.so.2 cannot be loaded: ") + (dlerror() ? dlerror() : "?");
            return a;
        }
        a.CommInitAll = reinterpret_cast<decltype(a.CommInitAll)>(dlsym(h, "ncclCommInitAll"));
        a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
        a.GroupStart = reinterpret_cast<decltype(a.GroupStart)>(dlsym(h, "ncclGroupStart"));
        a.GroupEnd = reinterpret_cast<decltype(a.GroupEnd)>(dlsym(h, "ncclGroupEnd"));
        a.AllGather = reinterpret_cast<decltype(a.AllGather)>(dlsym(h, "ncclAllGather"));
        a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
        a.GetVersion = reinterpret_cast<decltype(a.GetVersion)>(dlsym(h, "ncclGetVersion"));
        a.ok = a.CommInitAll && a.CommDestroy && a.GroupStart && a.GroupEnd && a.AllGather && a.GetErrorString;
        if (!a.ok) a.origin += " (required symbols missing)";
        return a;
    }();
    return api;
}

struct Shard {
    int device = 0;
    dawn_index *idx = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    // per-call device buffers (grown on demand)
    float *d_q = nullptr;
    uint8_t *d_block = nullptr;
    uint8_t *d_gather = nullptr;  // [G][block] receive buffer of the all-gather on this device
    size_t gather_cap = 0;
    ncclComm_t comm = nullptr;
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;  // device time of the local search
    float search_ms = 0.f;
    uint32_t *d_flags = nullptr;
    uint32_t *h_flags = nullptr;  // pinned
    float *h_q = nullptr;         // pinned copy of the queries for this device
    size_t q_cap = 0, block_cap = 0;
    // worker thread
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::function<int()> job;
    bool has_job = false, stop = false;
    int rc = 0;
    std::string err;
    bool job_done = false;
};

size_t block_bytes(size_t batch, size_t k) { return (batch * k * 12 + batch * 4 + 15) / 16 * 16; }

}  // namespace

struct dawn_multi {
    std::vector<Shard *> shards;
    std::mutex mu;
    uint32_t scalar = DAWN_SCALAR_F16;
    // device 0 side
    uint8_t *d_gather = nullptr, *d_out = nullptr;
    uint8_t *h_out = nullptr;
    size_t gather_cap = 0, out_cap = 0;
    size_t next_shard = 0;  // round-robin cursor for add
    bool nccl_ready = false;   // communicators exist (distinct devices, more than one shard)
    int exchange = 0;          // 0 = auto (NCCL when ready), 1 = peer copies, 2 = NCCL (error if not ready)
    cudaEvent_t ev_x0 = nullptr, ev_x1 = nullptr;  // device time of exchange + merge on the first device
    double last_search_ms = 0, last_exchange_ms = 0;
    uint64_t searches = 0, nccl_exchanges = 0, peer_exchanges = 0, reruns = 0;
};

namespace {

void worker_loop(Shard *s) {
    cudaSetDevice(s->device);
    std::unique_lock<std::mutex> lk(s->mu);
    while (true) {
        s->cv.wait(lk, [&] { return s->has_job || s->stop; });
        if (s->stop) return;
        auto job = s->job;
        lk.unlock();
        g_multi_err.clear();
        int rc = job();
        std::string err = rc ? (g_multi_err.empty() ? std::string(dawn_last_error()) : g_multi_err) : std::string();
        lk.lock();
        s->rc = rc;
        s->err = err;
        s->has_job = false;
        s->job_done = true;
        s->cv.notify_all();
    }
}

void submit(Shard *s, std::function<int()> job) {
    std::lock_guard<std::mutex> lk(s->mu);
    s->job = std::move(job);
    s->has_job = true;
    s->job_done = false;
    s->cv.notify_all();
}

int wait(Shard *s) {
    std::unique_lock<std::mutex> lk(s->mu);
    s->cv.wait(lk, [&] { return s->job_done; });
    if (s->rc) g_multi_err = s->err;
    return s->rc;
}

int run_all(dawn_multi *m, const std::function<int(Shard *, size_t)> &fn) {
    for (size_t g = 0; g < m->shards.size(); g++) {
        Shard *s = m->shards[g];
        submit(s, [=] { return fn(s, g); });
    }
    int rc = DAWN_OK;
    for (Shard *s : m->shards) {
        int r = wait(s);
        if (r && !rc) rc = r;
    }
    return rc;
}

int cuda_fail(cudaError_t e, const char *what) {
    g_multi_err = std::string(what) + ": " + cudaGetErrorString(e);
    return DAWN_ERR_CUDA;
}

}  // namespace

extern "C" {

const char *dawn_multi_last_error(void) { return g_multi_err.c_str(); }

int dawn_multi_create(const int *devices, size_t n_devices, uint32_t scalar, dawn_multi **out) {
    if (!devices || n_devices == 0 || n_devices > 64 || !out) return DAWN_ERR_INVALID;
    dawn_multi *m = new (std::nothrow) dawn_multi();
    if (!m) return DAWN_ERR_INTERNAL;
    m->scalar = scalar;
    for (size_t g = 0; g < n_devices; g++) {
        Shard *s = new Shard();
        s->device = devices[g];
        dawn_options o{};
        o.dimensions = DAWN_DIMENSIONS;
        o.scalar = scalar;
        o.device = devices[g];
        int rc = dawn_index_create(&o, &s->idx);
        if (rc == DAWN_OK) {
            cudaError_t e = cudaSetDevice(s->device);
            if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->done, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreate(&s->ev_a);
            if (e == cudaSuccess) e = cudaEventCreate(&s->ev_b);
            if (e != cudaSuccess) rc = cuda_fail(e, "shard setup");
        } else {
            g_multi_err = dawn_last_error();
        }
        m->shards.push_back(s);
        if (rc != DAWN_OK) {
            dawn_multi_free(m);
            return rc;
        }
        s->th = std::thread(worker_loop, s);
    }
    {
        cudaSetDevice(m->shards[0]->device);
        cudaEventCreate(&m->ev_x0);
        cudaEventCreate(&m->ev_x1);
    }
    // One NCCL communicator per shard, all in this process.  NCCL refuses a device listed twice;
    // such handles (tests on a one-GPU box) keep the peer-copy exchange.
    bool distinct = n_devices > 1;
    for (size_t a = 0; a < n_devices && distinct; a++)
        for (size_t b = a + 1; b < n_devices; b++)
            if (devices[a] == devices[b]) distinct = false;
    if (distinct && !getenv("DAWN_MULTI_NO_NCCL")) {
        const NcclApi &nccl = nccl_api();
        if (!nccl.ok) {  // several GPUs were asked for and the exchange they need is missing: fail loudly, no silent peer-copy fallback
            g_multi_err = "NCCL is required for a multi-GPU handle: " + nccl.origin;
            dawn_multi_free(m);
            return DAWN_ERR_CUDA;
        }
        std::vector<ncclComm_t> comms(n_devices);
        ncclResult_t nr = nccl.CommInitAll(comms.data(), (int)n_devices, devices);
        if (nr != ncclSuccess) {
            g_multi_err = std::string("ncclCommInitAll: ") + nccl.GetErrorString(nr);
            dawn_multi_free(m);
            return DAWN_ERR_CUDA;
        }
        for (size_t g = 0; g < n_devices; g++) m->shards[g]->comm = comms[g];
        m->nccl_ready = true;
    }
    *out = m;
    return DAWN_OK;
}

void dawn_multi_free(dawn_multi *m) {
    if (!m) return;
    const int dev0 = m->shards.empty() ? -1 : m->shards[0]->device;  // the shards are deleted below
    for (Shard *s : m->shards) {
        if (s->th.joinable()) {
            {
                std::lock_guard<std::mutex> lk(s->mu);
                s->stop = true;
            }
            s->cv.notify_all();
            s->th.join();
        }
        cudaSetDevice(s->device);
        if (s->comm) nccl_api().CommDestroy(s->comm);
        if (s->ev_a) cudaEventDestroy(s->ev_a);
        if (s->ev_b) cudaEventDestroy(s->ev_b);
        cudaFree(s->d_gather);
        cudaFree(s->d_q);
        cudaFree(s->d_block);
        cudaFree(s->d_flags);
        cudaFreeHost(s->h_flags);
        cudaFreeHost(s->h_q);
        if (s->done) cudaEventDestroy(s->done);
        if (s->stream) cudaStreamDestroy(s->stream);
        dawn_index_free(s->idx);
        delete s;
    }
    if (dev0 >= 0) cudaSetDevice(dev0);
    if (m->ev_x0) cudaEventDestroy(m->ev_x0);
    if (m->ev_x1) cudaEventDestroy(m->ev_x1);
    cudaFree(m->d_gather);
    cudaFree(m->d_out);
    cudaFreeHost(m->h_out);
    cudaGetLastError();
    delete m;
}

size_t dawn_multi_shards(const dawn_multi *m) { return m ? m->shards.size() : 0; }

size_t dawn_multi_size(const dawn_multi *m) {
    size_t n = 0;
    if (m)
        for (Shard *s : m->shards) n += dawn_index_size(s->idx);
    return n;
}

size_t dawn_multi_capacity(const dawn_multi *m) {
    size_t n = 0;
    if (m)
        for (Shard *s : m->shards) n += dawn_index_capacity(s->idx);
    return n;
}

// Capacity is split evenly over the shards.
int dawn_multi_reserve(dawn_multi *m, size_t n_total) {
    if (!m) return DAWN_ERR_INVALID;
    std::lock_guard<std::mutex> lk(m->mu);
    const size_t per = (n_total + m->shards.size() - 1) / m->shards.size();
    for (Shard *s : m->shards) {
        int rc = dawn_index_reserve(s->idx, per);
        if (rc) {
            g_multi_err = dawn_last_error();
            return rc;
        }
    }
    return DAWN_OK;
}

// Appends go to the shards in blocks, round-robin, skipping full shards (labels travel with the
// vectors, so any placement gives the same answers).
int dawn_multi_add_batch(dawn_multi *m, const uint64_t *labels, const float *vectors, size_t n) {
    if (!m || (n && (!labels || !vectors))) return DAWN_ERR_INVALID;
    std::lock_guard<std::mutex> lk(m->mu);
    const size_t kBlock = 4096;
    size_t done = 0;
    while (done < n) {
        size_t tries = 0;
        Shard *s = nullptr;
        size_t room = 0;
        while (tries < m->shards.size()) {
            s = m->shards[m->next_shard % m->shards.size()];
            room = dawn_index_capacity(s->idx) - dawn_index_size(s->idx);
            if (room > 0) break;
            m->next_shard++;
            tries++;
        }
        if (room == 0) {
            g_multi_err = "add exceeds the reserved capacity of every shard: reserve first";
            return DAWN_ERR_CAPACITY;
        }
        size_t take = n - done < kBlock ? n - done : kBlock;
        if (take > room) take = room;
        int rc = dawn_index_add_batch(s->idx, labels + done, vectors + done * DAWN_DIMENSIONS, take);
        if (rc) {
            g_multi_err = dawn_last_error();
            return rc;
        }
        done += take;
        m->next_shard++;
    }
    return DAWN_OK;
}

int dawn_multi_add(dawn_multi *m, uint64_t label, const float *vector384) {
    return dawn_multi_add_batch(m, &label, vector384, 1);
}

// Synthetic corpus rows [first_row, first_row+n) split into contiguous id ranges, one per shard.
int dawn_multi_add_synthetic(dawn_multi *m, uint64_t seed, uint64_t first_row, size_t n) {
    if (!m) return DAWN_ERR_INVALID;
    std::lock_guard<std::mutex> lk(m->mu);
    const size_t G = m->shards.size();
    const size_t per = (n + G - 1) / G;
    return run_all(m, [=](Shard *s, size_t g) -> int {
        const size_t a = g * per < n ? g * per : n;
        const size_t cnt = a + per < n ? per : n - a;
        if (cnt == 0) return DAWN_OK;
        return dawn_index_add_synthetic(s->idx, seed, first_row + a, cnt);
    });
}

// Adds place labels on any shard, so every shard runs the remove (concurrently); the counts are summed.
int dawn_multi_remove_batch(dawn_multi *m, const uint64_t *labels, size_t n, size_t *removed_out) {
    if (removed_out) *removed_out = 0;
    if (!m || (n && !labels)) {
        g_multi_err = !m ? "null multi handle" : "labels is null";
        return DAWN_ERR_INVALID;
    }
    if (n == 0) return DAWN_OK;
    std::lock_guard<std::mutex> lk(m->mu);
    std::vector<size_t> removed(m->shards.size(), 0);
    size_t *counts = removed.data();
    int rc = run_all(m, [=](Shard *s, size_t g) -> int { return dawn_index_remove_batch(s->idx, labels, n, counts + g); });
    // a shard that failed reports 0; the others have removed their rows, and the count says so even when rc != 0
    if (removed_out)
        for (size_t r : removed) *removed_out += r;
    return rc;
}

int dawn_multi_remove(dawn_multi *m, uint64_t label, size_t *removed_out) {
    return dawn_multi_remove_batch(m, &label, 1, removed_out);
}

// distance_limit (NaN = none): every shard pushes the limit down into its kernels and cuts its counts on the device, so
// only hits with distance < limit are exchanged and merged (UdpPacket::Search.distance_limit, src/net/udp_packets.rs:29-39;
// filter src/net/udp_service.rs:196-199).
int dawn_multi_search_batch_limit(dawn_multi *m, const float *queries, size_t batch, size_t k, float distance_limit,
                                  uint64_t *labels_out, float *distances_out, size_t *counts_out) {
    if (!m || !queries || !counts_out || (k && (!labels_out || !distances_out))) return DAWN_ERR_INVALID;
    if (batch == 0) return DAWN_OK;
    if (k == 0) {
        for (size_t b = 0; b < batch; b++) counts_out[b] = 0;
        return DAWN_OK;
    }
    if (k > DAWN_MAX_K || m->shards.size() * k > 1024) {
        g_multi_err = "k too large for this many shards (shards * k must be <= 1024)";
        return DAWN_ERR_INVALID;
    }
    std::lock_guard<std::mutex> lk(m->mu);
    const size_t G = m->shards.size();
    const size_t bb = block_bytes(batch, k);
    const size_t off_d = batch * k * 8, off_c = off_d + batch * k * 4;
    if (m->exchange == 2 && !m->nccl_ready) {
        g_multi_err = "exchange = nccl requested but no communicator exists (one shard, or a device listed twice)";
        return DAWN_ERR_INVALID;
    }
    // auto: the all-gather for real batches; for a handful of queries the blocks are a few hundred bytes and one peer copy per
    // shard into the first device is ~60 us quicker than eight communicators' worth of collective launches (measured on
    // 8 B200: 18 us against 84 us for exchange + merge at batch 1, profiles/r02_front_multi_k10_8gpu.json)
    const bool use_nccl = m->nccl_ready && (m->exchange == 2 || (m->exchange == 0 && bb > 16384));
    Shard *s0 = m->shards[0];
    cudaError_t e = cudaSetDevice(s0->device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    if (!use_nccl && G * bb > m->gather_cap) {
        cudaFree(m->d_gather);
        m->gather_cap = 0;
        if ((e = cudaMalloc(&m->d_gather, G * bb)) != cudaSuccess) return cuda_fail(e, "cudaMalloc gather");
        m->gather_cap = G * bb;
    }
    if (bb > m->out_cap) {
        cudaFree(m->d_out);
        cudaFreeHost(m->h_out);
        m->out_cap = 0;
        if ((e = cudaMalloc(&m->d_out, bb)) != cudaSuccess) return cuda_fail(e, "cudaMalloc out");
        if ((e = cudaMallocHost(&m->h_out, bb)) != cudaSuccess) return cuda_fail(e, "cudaMallocHost out");
        m->out_cap = bb;
    }
    uint8_t *d_gather_peer = m->d_gather;
    const int dev0 = s0->device;
    std::atomic<uint64_t> reruns{0};

    // every shard: H2D queries, local exact top-k into a packed block; then either its peer copy into the
    // first device's gather buffer, or nothing (the all-gather is issued for all shards as one group below)
    int rc = run_all(m, [=, &reruns](Shard *s, size_t g) -> int {
        cudaError_t ce;
        if (batch > s->q_cap) {
            cudaFree(s->d_q);
            cudaFree(s->d_flags);
            cudaFreeHost(s->h_flags);
            cudaFreeHost(s->h_q);
            s->q_cap = 0;
            const size_t cap = batch < 64 ? 64 : batch;
            if ((ce = cudaMalloc(&s->d_q, cap * DAWN_DIMENSIONS * sizeof(float))) != cudaSuccess) return cuda_fail(ce, "cudaMalloc q");
            if ((ce = cudaMalloc(&s->d_flags, cap * sizeof(uint32_t))) != cudaSuccess) return cuda_fail(ce, "cudaMalloc flags");
            if ((ce = cudaMallocHost(&s->h_flags, cap * sizeof(uint32_t))) != cudaSuccess) return cuda_fail(ce, "cudaMallocHost flags");
            if ((ce = cudaMallocHost(&s->h_q, cap * DAWN_DIMENSIONS * sizeof(float))) != cudaSuccess) return cuda_fail(ce, "cudaMallocHost q");
            s->q_cap = cap;
        }
        if (bb > s->block_cap) {
            cudaFree(s->d_block);
            s->block_cap = 0;
            if ((ce = cudaMalloc(&s->d_block, bb)) != cudaSuccess) return cuda_fail(ce, "cudaMalloc block");
            s->block_cap = bb;
        }
        if (use_nccl && G * bb > s->gather_cap) {
            cudaFree(s->d_gather);
            s->gather_cap = 0;
            if ((ce = cudaMalloc(&s->d_gather, G * bb)) != cudaSuccess) return cuda_fail(ce, "cudaMalloc gather");
            s->gather_cap = G * bb;
        }
        memcpy(s->h_q, queries, batch * DAWN_DIMENSIONS * sizeof(float));
        if ((ce = cudaMemcpyAsync(s->d_q, s->h_q, batch * DAWN_DIMENSIONS * sizeof(float), cudaMemcpyHostToDevice, s->stream)) != cudaSuccess)
            return cuda_fail(ce, "H2D queries");
        if ((ce = cudaMemsetAsync(s->d_block, 0, bb, s->stream)) != cudaSuccess) return cuda_fail(ce, "memset block");
        cudaEventRecord(s->ev_a, s->stream);
        int r = dawn_index_search_device_limit(s->idx, s->d_q, batch, k, distance_limit, reinterpret_cast<uint64_t *>(s->d_block),
                                         reinterpret_cast<float *>(s->d_block + off_d),
                                         reinterpret_cast<uint32_t *>(s->d_block + off_c), s->d_flags, s->stream);
        if (r) return r;
        cudaEventRecord(s->ev_b, s->stream);
        if ((ce = cudaMemcpyAsync(s->h_flags, s->d_flags, batch * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream)) != cudaSuccess)
            return cuda_fail(ce, "D2H flags");
        if ((ce = cudaStreamSynchronize(s->stream)) != cudaSuccess) return cuda_fail(ce, "shard sync");
        cudaEventElapsedTime(&s->search_ms, s->ev_a, s->ev_b);
        // queries this shard could not certify: exact re-run through the host API, patched into the block
        if (dawn_index_size(s->idx) > 0) {
            std::vector<uint64_t> l(k);
            std::vector<float> d(k);
            for (size_t b = 0; b < batch; b++) {
                if (s->h_flags[b] & 1u) continue;
                size_t cnt = 0;
                r = dawn_index_search_limit(s->idx, queries + b * DAWN_DIMENSIONS, k, distance_limit, l.data(), d.data(), &cnt);
                if (r) return r;
                reruns++;
                uint32_t c32 = (uint32_t)cnt;
                cudaMemcpyAsync(s->d_block + b * k * 8, l.data(), cnt * 8, cudaMemcpyHostToDevice, s->stream);
                cudaMemcpyAsync(s->d_block + off_d + b * k * 4, d.data(), cnt * 4, cudaMemcpyHostToDevice, s->stream);
                cudaMemcpyAsync(s->d_block + off_c + b * 4, &c32, 4, cudaMemcpyHostToDevice, s->stream);
                if ((ce = cudaStreamSynchronize(s->stream)) != cudaSuccess) return cuda_fail(ce, "patch sync");
            }
        }
        if (!use_nccl) {
            // one message per shard over NVLink into the first device's gather buffer
            if ((ce = cudaMemcpyPeerAsync(d_gather_peer + g * bb, dev0, s->d_block, s->device, bb, s->stream)) != cudaSuccess)
                return cuda_fail(ce, "peer copy");
            if ((ce = cudaStreamSynchronize(s->stream)) != cudaSuccess) return cuda_fail(ce, "peer sync");
        }
        return DAWN_OK;
    });
    if (rc) return rc;
    m->reruns += reruns;
    m->searches++;
    double smax = 0;
    for (Shard *s : m->shards) smax = s->search_ms > smax ? s->search_ms : smax;
    m->last_search_ms = smax;

    if ((e = cudaSetDevice(dev0)) != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    cudaEventRecord(m->ev_x0, s0->stream);
    const uint8_t *d_gather = d_gather_peer;
    if (use_nccl) {
        // THE exchange: one all-gather of the packed blocks, issued for every shard's communicator as one group
        // (every shard's stream is idle here, so the collective starts at once on all GPUs)
        const NcclApi &nccl = nccl_api();
        ncclResult_t nr = nccl.GroupStart();
        for (size_t g = 0; g < G && nr == ncclSuccess; g++) {
            Shard *s = m->shards[g];
            nr = nccl.AllGather(s->d_block, s->d_gather, bb, ncclUint8, s->comm, s->stream);
        }
        ncclResult_t ne = nccl.GroupEnd();
        if (nr == ncclSuccess) nr = ne;
        if (nr != ncclSuccess) {
            g_multi_err = std::string("ncclAllGather: ") + nccl.GetErrorString(nr);
            return DAWN_ERR_CUDA;
        }
        m->nccl_exchanges++;
        d_gather = s0->d_gather;
        cudaSetDevice(dev0);
    } else {
        m->peer_exchanges++;
    }
    // device-side merge on the first device, then one D2H of the merged block
    rc = dawn_merge_results_device(dev0, reinterpret_cast<const uint64_t *>(d_gather), reinterpret_cast<const float *>(d_gather + off_d),
                                   reinterpret_cast<const uint32_t *>(d_gather + off_c), G, bb, batch, k,
                                   reinterpret_cast<uint64_t *>(m->d_out), reinterpret_cast<float *>(m->d_out + off_d),
                                   reinterpret_cast<uint32_t *>(m->d_out + off_c), s0->stream);
    if (rc) {
        g_multi_err = dawn_last_error();
        return rc;
    }
    cudaEventRecord(m->ev_x1, s0->stream);
    if ((e = cudaMemcpyAsync(m->h_out, m->d_out, bb, cudaMemcpyDeviceToHost, s0->stream)) != cudaSuccess) return cuda_fail(e, "D2H out");
    if ((e = cudaStreamSynchronize(s0->stream)) != cudaSuccess) return cuda_fail(e, "final sync");
    if (use_nccl)  // the other shards' receive buffers are reused by the next call
        for (size_t g = 1; g < G; g++) {
            cudaSetDevice(m->shards[g]->device);
            if ((e = cudaStreamSynchronize(m->shards[g]->stream)) != cudaSuccess) return cuda_fail(e, "all-gather sync");
        }
    float xms = 0.f;
    cudaEventElapsedTime(&xms, m->ev_x0, m->ev_x1);
    m->last_exchange_ms = xms;
    const uint32_t *cnt = reinterpret_cast<const uint32_t *>(m->h_out + off_c);
    for (size_t b = 0; b < batch; b++) {
        counts_out[b] = cnt[b];
        memcpy(labels_out + b * k, m->h_out + b * k * 8, cnt[b] * 8);
        memcpy(distances_out + b * k, m->h_out + off_d + b * k * 4, cnt[b] * 4);
    }
    return DAWN_OK;
}

// "exchange": 0 = auto (NCCL all-gather when communicators exist), 1 = peer copies, 2 = NCCL or fail.
int dawn_multi_set_option(dawn_multi *m, const char *key, int64_t value) {
    if (!m || !key) return DAWN_ERR_INVALID;
    std::lock_guard<std::mutex> lk(m->mu);
    if (!strcmp(key, "exchange")) {
        if (value < 0 || value > 2) return DAWN_ERR_INVALID;
        m->exchange = (int)value;
        return DAWN_OK;
    }
    // everything else is a per-shard index option
    for (Shard *s : m->shards) {
        int rc = dawn_index_set_option(s->idx, key, value);
        if (rc) {
            g_multi_err = dawn_last_error();
            return rc;
        }
    }
    return DAWN_OK;
}

int dawn_multi_get_stats(dawn_multi *m, dawn_multi_stats *out) {
    if (!m || !out) return DAWN_ERR_INVALID;
    std::lock_guard<std::mutex> lk(m->mu);
    out->searches = m->searches;
    out->nccl_exchanges = m->nccl_exchanges;
    out->peer_exchanges = m->peer_exchanges;
    out->exact_reruns = m->reruns;
    out->last_search_ms = m->last_search_ms;
    out->last_exchange_ms = m->last_exchange_ms;
    out->nccl_ready = m->nccl_ready ? 1 : 0;
    out->kernel_launches = 0;
    for (Shard *s : m->shards) {
        dawn_profile p{};
        if (dawn_index_get_profile(s->idx, &p, 0) == DAWN_OK) out->kernel_launches += p.kernel_launches;
    }
    out->kernel_launches += m->searches + m->nccl_exchanges * m->shards.size();  // merge kernel + NCCL's kernels
    return DAWN_OK;
}

int dawn_multi_search_batch(dawn_multi *m, const float *queries, size_t batch, size_t k, uint64_t *labels_out,
                            float *distances_out, size_t *counts_out) {
    return dawn_multi_search_batch_limit(m, queries, batch, k, NAN, labels_out, distances_out, counts_out);
}

int dawn_multi_search_limit(dawn_multi *m, const float *query384, size_t k, float distance_limit, uint64_t *labels_out,
                            float *distances_out, size_t *count_out) {
    return dawn_multi_search_batch_limit(m, query384, 1, k, distance_limit, labels_out, distances_out, count_out);
}

int dawn_multi_search(dawn_multi *m, const float *query384, size_t k, uint64_t *labels_out, float *distances_out,
                      size_t *count_out) {
    return dawn_multi_search_batch(m, query384, 1, k, labels_out, distances_out, count_out);
}

}  // extern "C"
