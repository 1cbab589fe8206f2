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
#include <fcntl.h>
#include <nccl.h>  // types and prototypes only: the library is bound at run time, see NcclApi
#include <sys/stat.h>
#include <unistd.h>

#include "../../include/dawn_index.h"
#include "persist.cuh"

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
    // Every call takes `mu` except save; the calls that change what the shards hold (save, load, add*, remove, reserve,
    // set_option) first take `writer_mu`.  So a save, which holds writer_mu alone, keeps the shards still while it writes
    // them out, and searches and gets go on meanwhile.
    std::mutex writer_mu;
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

// fn for every shard at once, each on a thread of its own, for the calls that run without mu (save, and the fill of a
// load): the shard workers serve one caller at a time, the one holding mu, so those calls must not queue on them.
int run_parallel(dawn_multi *m, const std::function<int(Shard *, size_t)> &fn) {
    const size_t G = m->shards.size();
    std::vector<int> rcs(G, DAWN_OK);
    std::vector<std::string> errs(G);
    std::vector<std::thread> threads;
    for (size_t g = 0; g < G; g++)
        threads.emplace_back([&, g] {
            Shard *s = m->shards[g];
            g_multi_err.clear();
            cudaError_t e = cudaSetDevice(s->device);
            rcs[g] = e != cudaSuccess ? cuda_fail(e, "cudaSetDevice") : fn(s, g);
            if (rcs[g]) errs[g] = g_multi_err.empty() ? std::string(dawn_last_error()) : g_multi_err;
        });
    for (std::thread &t : threads) t.join();
    for (size_t g = 0; g < G; g++)
        if (rcs[g]) {
            g_multi_err = errs[g];
            return rcs[g];
        }
    return DAWN_OK;
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
    std::lock_guard<std::mutex> wk(m->writer_mu);
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
    std::lock_guard<std::mutex> wk(m->writer_mu);
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
    std::lock_guard<std::mutex> wk(m->writer_mu);
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
    std::lock_guard<std::mutex> wk(m->writer_mu);
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
    std::lock_guard<std::mutex> wk(m->writer_mu);
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

// ---- persistence: one file for the whole handle (include/dawn_index.h, DESIGN.md section 6) ----------------------------

}  // extern "C"

namespace {

using dawn::SectionRef;

constexpr uint64_t kMultiHeaderBytes = 4096;  // also the alignment of every section: concurrent writers never share a page
constexpr size_t kMaxShardRows = 0xFFFFFFF0ull;  // a shard holds fewer rows than this (grow_physical's limit)
constexpr uint64_t kMaxFileRows = 1ull << 40;    // row counts beyond this cannot come from a real file

struct MultiHeader {  // the first 32 bytes of a DAWNMULT file; uint64 rows[G] follow, then zeros up to kMultiHeaderBytes
    char magic[8];    // "DAWNMULT"
    uint32_t version, scalar, dims, shards;
    uint64_t next_shard;
};
static_assert(sizeof(MultiHeader) == 32, "file layout");

// Sets off[g] to section g's start; returns the file length (the end of the last section).
uint64_t multi_layout(uint32_t scalar, const std::vector<uint64_t> &rows, std::vector<uint64_t> &off) {
    uint64_t end = kMultiHeaderBytes;
    off.resize(rows.size());
    for (size_t g = 0; g < rows.size(); g++) {
        off[g] = (end + kMultiHeaderBytes - 1) / kMultiHeaderBytes * kMultiHeaderBytes;
        end = off[g] + rows[g] * sizeof(uint64_t) + dawn::section_payload_bytes(scalar, rows[g]);
    }
    return end;
}

// The sections of a DAWNMULT file, or of a DAWNB200 single-index file (one section, cursor 0).  Everything is checked
// against the handle's storage type and against the file's length before any device work.
bool read_sections(int fd, uint32_t scalar, std::vector<SectionRef> *secs, uint64_t *cursor, std::string *why) {
    unsigned char head[32];
    struct stat st;
    if (fstat(fd, &st) != 0 || !dawn::pread_all(fd, head, sizeof head, 0)) {
        *why = "shorter than a header";
        return false;
    }
    uint32_t version, file_scalar, dims;
    memcpy(&version, head + 8, 4);
    memcpy(&file_scalar, head + 12, 4);
    memcpy(&dims, head + 16, 4);
    uint64_t want = 0;
    if (!memcmp(head, "DAWNB200", 8) || !memcmp(head, "DAWNMULT", 8)) {
        if (version != 1 || file_scalar != scalar || dims != DAWN_DIMENSIONS) {
            *why = "version, storage type or dimensions differ from this handle's";
            return false;
        }
    } else {
        *why = "not a libdawn_b200 index file";
        return false;
    }
    if (!memcmp(head, "DAWNB200", 8)) {
        uint64_t size;
        memcpy(&size, head + 24, 8);
        if (size > kMaxFileRows) {
            *why = "row count out of range";
            return false;
        }
        secs->assign(1, SectionRef{sizeof head, size});
        *cursor = 0;
        want = sizeof head + size * sizeof(uint64_t) + dawn::section_payload_bytes(scalar, size);
    } else {
        MultiHeader h;
        memcpy(&h, head, sizeof h);
        if (h.shards < 1 || h.shards > 64 || h.next_shard >= h.shards) {
            *why = "shard count or add cursor out of range";
            return false;
        }
        std::vector<uint64_t> rows(h.shards), off;
        if (!dawn::pread_all(fd, rows.data(), rows.size() * sizeof(uint64_t), sizeof h)) {
            *why = "header cut short";
            return false;
        }
        for (uint64_t r : rows)
            if (r > kMaxFileRows) {
                *why = "row count out of range";
                return false;
            }
        want = multi_layout(scalar, rows, off);
        secs->clear();
        for (size_t g = 0; g < rows.size(); g++) secs->push_back(SectionRef{off[g], rows[g]});
        *cursor = h.next_shard;
    }
    if ((uint64_t)st.st_size != want) {
        *why = "file length " + std::to_string((long long)st.st_size) + " differs from the " + std::to_string(want) +
               " bytes its header implies";
        return false;
    }
    return true;
}

int io_fail(const char *path, const std::string &why) {
    g_multi_err = std::string(path) + ": " + why;
    return DAWN_ERR_IO;
}

}  // namespace

extern "C" {

// Header, then each shard's section written by a thread of its own (pwrite at its own page-aligned offset), to path.tmp,
// renamed when every section is on disk.  Holds only writer_mu: adds and removes wait, searches and gets go on.
int dawn_multi_save(dawn_multi *m, const char *path) {
    if (!m || !path) {
        g_multi_err = !m ? "null multi handle" : "path is null";
        return DAWN_ERR_INVALID;
    }
    std::lock_guard<std::mutex> wk(m->writer_mu);
    const size_t G = m->shards.size();
    std::vector<uint64_t> rows(G), off;
    uint64_t *r = rows.data();
    int rc = run_parallel(m, [=](Shard *s, size_t g) -> int { return dawn::section_prepare(s->idx, false, r + g); });
    if (rc) return rc;
    const uint64_t len = multi_layout(m->scalar, rows, off);
    std::vector<unsigned char> head(kMultiHeaderBytes, 0);
    MultiHeader h{};
    memcpy(h.magic, "DAWNMULT", 8);
    h.version = 1;
    h.scalar = m->scalar;
    h.dims = DAWN_DIMENSIONS;
    h.shards = (uint32_t)G;
    h.next_shard = m->next_shard % G;
    memcpy(head.data(), &h, sizeof h);
    memcpy(head.data() + sizeof h, rows.data(), G * sizeof(uint64_t));
    const std::string tmp = std::string(path) + ".tmp";
    const int fd = open(tmp.c_str(), O_WRONLY | O_CREAT | O_TRUNC | O_CLOEXEC, 0666);
    if (fd < 0) return io_fail(tmp.c_str(), "cannot open for writing");
    // the gaps between sections are holes of the right length, read back as the zero padding
    if (ftruncate(fd, (off_t)len) != 0 || !dawn::pwrite_all(fd, head.data(), head.size(), 0)) {
        rc = io_fail(tmp.c_str(), "short write");
    } else {
        const uint64_t *o = off.data();
        rc = run_parallel(m, [=](Shard *s, size_t g) -> int { return dawn::section_write(s->idx, fd, o[g], r[g]); });
    }
    const int frc = dawn::finish_file(fd, tmp.c_str(), path, rc);
    if (frc != rc) g_multi_err = dawn_last_error();
    return frc;
}

// Phase 1 fills every shard at once (run_parallel); phase 2 publishes all of them under mu, so no search sees old and new shards
// mixed, and a failure of any shard leaves the handle as it was.  Same shard count: section g -> shard g and the add cursor
// is restored.  Otherwise the sections are concatenated and shard g gets rows [g P, min(N, (g+1) P)), P = ceil(N / G),
// cursor 0.
int dawn_multi_load(dawn_multi *m, const char *path) {
    if (!m || !path) {
        g_multi_err = !m ? "null multi handle" : "path is null";
        return DAWN_ERR_INVALID;
    }
    std::lock_guard<std::mutex> wk(m->writer_mu);
    const size_t G = m->shards.size();
    const int fd = open(path, O_RDONLY | O_CLOEXEC);
    if (fd < 0) return io_fail(path, "cannot open");
    std::vector<SectionRef> secs;
    uint64_t cursor = 0;
    std::string why;
    if (!read_sections(fd, m->scalar, &secs, &cursor, &why)) {
        close(fd);
        return io_fail(path, why);
    }
    uint64_t total = 0;
    for (const SectionRef &sr : secs) total += sr.rows;
    std::vector<uint64_t> first(G), count(G);
    const uint64_t per = (total + G - 1) / G;
    for (size_t g = 0, at = 0; g < G; g++) {
        if (secs.size() == G) {
            first[g] = at;
            count[g] = secs[g].rows;
            at += secs[g].rows;
        } else {
            first[g] = g * per < total ? g * per : total;
            count[g] = first[g] + per < total ? per : total - first[g];
        }
        if (count[g] >= kMaxShardRows) {
            close(fd);
            return io_fail(path, "more rows per shard than one GPU's index holds");
        }
    }
    if (secs.size() != G) cursor = 0;
    const bool was_empty = dawn_multi_size(m) == 0;
    std::vector<dawn::Fill> fills(G);
    dawn::Fill *fp = fills.data();
    const SectionRef *sp = secs.data();
    const size_t n_secs = secs.size();
    const uint64_t *fi = first.data(), *co = count.data();
    int rc = run_parallel(m, [=](Shard *s, size_t g) -> int {
        uint64_t held = 0;
        int r = dawn::section_prepare(s->idx, false, &held);  // flushes staged adds: they belong to the old contents
        if (r) return r;
        return dawn::fill_rows(s->idx, fd, path, sp, n_secs, fi[g], co[g], was_empty, fp + g);
    });
    close(fd);
    if (rc) {
        for (size_t g = 0; g < G; g++) dawn::fill_discard(m->shards[g]->idx, &fills[g]);
        return rc;
    }
    std::lock_guard<std::mutex> lk(m->mu);
    for (size_t g = 0; g < G; g++) dawn::fill_commit(m->shards[g]->idx, &fills[g]);
    m->next_shard = cursor;
    return DAWN_OK;
}

// Every shard looks the label up at once; the lowest-index shard holding it answers (the copy the merge keeps).
int dawn_multi_get(dawn_multi *m, uint64_t label, float *out384) {
    if (!m || !out384) {
        g_multi_err = !m ? "null multi handle" : "output is null";
        return DAWN_ERR_INVALID;
    }
    std::lock_guard<std::mutex> lk(m->mu);
    const size_t G = m->shards.size();
    std::vector<float> vec(G * DAWN_DIMENSIONS);
    std::vector<int> rcs(G, DAWN_OK);
    std::vector<std::string> errs(G);
    float *v = vec.data();
    int *rp = rcs.data();
    std::string *ep = errs.data();
    run_all(m, [=](Shard *s, size_t g) -> int {
        rp[g] = dawn_index_get(s->idx, label, v + g * DAWN_DIMENSIONS);
        if (rp[g]) ep[g] = dawn_last_error();
        return DAWN_OK;
    });
    for (size_t g = 0; g < G; g++)
        if (rcs[g] != DAWN_OK && rcs[g] != DAWN_ERR_INVALID) {  // a CUDA error, not an absent label
            g_multi_err = errs[g];
            return rcs[g];
        }
    for (size_t g = 0; g < G; g++)
        if (rcs[g] == DAWN_OK) {
            memcpy(out384, v + g * DAWN_DIMENSIONS, DAWN_DIMENSIONS * sizeof(float));
            return DAWN_OK;
        }
    g_multi_err = "label " + std::to_string((unsigned long long)label) + " not found";
    return DAWN_ERR_INVALID;
}

int dawn_multi_get_i24(dawn_multi *m, uint64_t label, uint8_t *out1152) {
    if (!out1152) {
        g_multi_err = "output is null";
        return DAWN_ERR_INVALID;
    }
    float v[DAWN_DIMENSIONS];
    int rc = dawn_multi_get(m, label, v);
    if (rc != DAWN_OK) return rc;
    dawn_encode_i24(v, out1152);
    return DAWN_OK;
}

// dawn_index_verify on every shard: bad rows summed, the smallest norm over non-empty shards (0 if all are empty), the largest.
int dawn_multi_verify(dawn_multi *m, size_t *bad_rows_out, float *min_norm_out, float *max_norm_out) {
    if (!m) {
        g_multi_err = "null multi handle";
        return DAWN_ERR_INVALID;
    }
    std::lock_guard<std::mutex> lk(m->mu);
    const size_t G = m->shards.size();
    std::vector<size_t> bad(G, 0), rows(G, 0);
    std::vector<float> lo(G, 0.f), hi(G, 0.f);
    size_t *bp = bad.data(), *np = rows.data();
    float *lp = lo.data(), *hp = hi.data();
    int rc = run_all(m, [=](Shard *s, size_t g) -> int {
        int r = dawn_index_verify(s->idx, bp + g, lp + g, hp + g);
        np[g] = dawn_index_size(s->idx);
        return r;
    });
    if (rc) return rc;
    size_t sum = 0;
    float mn = 0.f, mx = 0.f;
    bool any = false;
    for (size_t g = 0; g < G; g++) {
        sum += bad[g];
        mx = hi[g] > mx ? hi[g] : mx;
        if (rows[g]) {
            mn = !any || lo[g] < mn ? lo[g] : mn;
            any = true;
        }
    }
    if (bad_rows_out) *bad_rows_out = sum;
    if (min_norm_out) *min_norm_out = mn;
    if (max_norm_out) *max_norm_out = mx;
    return DAWN_OK;
}

// The peer side of a remote search over the whole handle: decoded as dawn_index_search_i24 does.
int dawn_multi_search_i24(dawn_multi *m, const uint8_t *query1152, size_t k, int has_limit, float distance_limit,
                          uint64_t *labels_out, float *distances_out, size_t *count_out) {
    if (!m || !query1152) {
        g_multi_err = !m ? "null multi handle" : "query is null";
        return DAWN_ERR_INVALID;
    }
    float q[DAWN_DIMENSIONS];
    if (dawn_decode_i24(query1152, q) != DAWN_OK) {
        g_multi_err = "Embedding is not normalized";
        return DAWN_ERR_INVALID;
    }
    return dawn_multi_search_limit(m, q, k, has_limit ? distance_limit : NAN, labels_out, distances_out, count_out);
}

}  // extern "C"
