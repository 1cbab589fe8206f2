// finalize.cu -- K5 + K6: merge the per-CTA candidate lists, re-score the survivors in the
// reference's order of summation, and emit the final (label, distance) pairs.
//
// K5 is the device counterpart of BestResults (/root/reference/src/search/best_results.rs:44-79):
// keep the k best of many partial result sets.  Unlike BestResults the order is total and
// independent of arrival: (score desc, label asc, row asc).
// K6 recomputes each surviving candidate's score exactly like the reference's scalar code
// (src/search/vector.rs:128-134: `result += a[i]*b[i]` in index order, one f32 rounding for
// the multiply and one for the add), so the scores, the final order and the distances
// (1 - score) are bit-identical to oracle/dawn_oracle.c:dawn_oracle_search_f16.
// The scan only has to deliver a superset: k' = k + slack candidates whose approximate
// scores are within `eps` of the exact ones.  The certificate bit says the slack was
// provably enough: every row the scan dropped scored <= the weakest kept candidate, which
// is more than eps below the k-th exact score.
//
// One CTA per query; latency-bound (a few microseconds), negligible bytes.
#include "dawn_common.cuh"

namespace dawn {

#ifdef DAWN_SCAN_TRACE  // tools/scan_trace.cu only
__device__ unsigned long long g_fin_trace[16];
#define FIN_TRACE(slot)                                                       \
    do {                                                                      \
        if (threadIdx.x == 0 && blockIdx.x == 0) {                            \
            unsigned long long t_;                                            \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));            \
            g_fin_trace[slot] = t_;                                           \
        }                                                                     \
    } while (0)
#else
#define FIN_TRACE(slot) do { } while (0)
#endif

namespace {

constexpr int kFinThreads = 1024;     // merging 148 per-CTA lists (scan path)
constexpr int kFinThreadsSingle = 128;  // one pre-merged list per query (tensor-core path)
constexpr int kFinCapEntries = 4096;  // 64 KB of candidates in shared memory per round
constexpr int kFinItems = kFinCapEntries / kFinThreads;

struct FinSmem {
    alignas(16) float q[kDim];
    uint32_t warp_min[kMaxCand / 32];
    uint32_t n_valid;
    float kth_dist;
    uint32_t n_surv;
    float bound;
    float q_norm2;
    alignas(16) Cand s[1];  // kFinCapEntries entries when merging, kp entries for a single list
};
constexpr int kRowStrideF16 = kRowBytesF16 + 16;  // staged candidate rows: +16 B so that thread-per-row reads are conflict free
constexpr int kRowStrideI8 = kDim + 16;
// header + candidate area + staged rows of the kp survivors
// (rows are staged only when merging per-CTA lists: one CTA per query on an otherwise idle GPU; with one
// pre-merged list per query there are as many CTAs as queries and occupancy matters more)
inline size_t fin_smem_bytes(int entries, int kp, int scalar, bool stage_rows) {
    return sizeof(FinSmem) + (size_t)(entries - 1) * sizeof(Cand) +
           (stage_rows ? (size_t)kp * (scalar ? kRowStrideI8 : kRowStrideF16) : 0);
}

__device__ __forceinline__ bool dist_before(const Cand &a, const Cand &b) {
    if (a.score != b.score) return a.score < b.score;
    if (a.label != b.label) return a.label < b.label;
    return a.row < b.row;
}

// S holds n_lists sorted lists of length kp (sentinel padded); tree-merge them into list 0.
// Each entry finds its rank in the union of its pair by binary search in the partner list.
__device__ void merge_lists(Cand *S, int n_lists, int kp, int tid) {
    for (int stride = 1; stride < n_lists; stride <<= 1) {
        const int n_pairs = (n_lists - stride + 2 * stride - 1) / (2 * stride);
        const int n_items = n_pairs * 2 * kp;
        Cand e[kFinItems];
        int dst[kFinItems];
#pragma unroll
        for (int it = 0; it < kFinItems; it++) {
            const int i = tid + it * kFinThreads;
            dst[it] = -1;
            if (i < n_items) {
                const int pair = i / (2 * kp);
                const int within = i % (2 * kp);
                const int a = pair * 2 * stride;
                const bool in_a = within < kp;
                const int p = in_a ? within : within - kp;
                const Cand *own = S + (size_t)(in_a ? a : a + stride) * kp;
                const Cand *other = S + (size_t)(in_a ? a + stride : a) * kp;
                e[it] = own[p];
                int lo = 0, hi = kp;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (cand_better(other[mid], e[it])) lo = mid + 1;
                    else hi = mid;
                }
                const int rank = p + lo;
                if (rank < kp) dst[it] = a * kp + rank;
            }
        }
        __syncthreads();
#pragma unroll
        for (int it = 0; it < kFinItems; it++)
            if (dst[it] >= 0) S[dst[it]] = e[it];
        __syncthreads();
    }
}

// Fast K5 for many short lists.  The kp-th best of the lists' first ceil(kp/n_lists) entries is a lower
// bound on the kp-th best score overall (those prefix entries are distinct candidates), so only
// entries at or above it can be in the result: with 148 lists that is a few dozen out of thousands.
// The survivors are ranked by counting under the full order and land sorted in S[0..kp).
// Returns false (uniformly) when more than kSelSurvCap entries survive -- long runs of equal scores --
// and the caller falls back to the tree merge.
constexpr int kSelProbeMax = 512;
constexpr int kSelSurvCap = 1024;

// How many of arr[0..n) come before `me`: by Cand::score (descending if DESC, else ascending), equal scores by
// (label asc, row asc).  The loop compares scores only and is shared by 1 << shift adjacent lanes; the
// label / row tie-break is a second pass run only when an equal score was actually met.  `self_in` = 1 if
// `me` is itself an element of arr.  Every lane of the warp must call (shuffles); the result is valid on sub == 0.
template <bool DESC>
__device__ __forceinline__ int count_before(const Cand *arr, int n, const Cand &me, bool active, int sub, int shift,
                                            int self_in) {
    int before = 0, eq = 0;
    const float ms = me.score;
    if (active) {
#pragma unroll 8
        for (int j = sub; j < n; j += 1 << shift) {
            const float s = arr[j].score;
            before += (DESC ? s > ms : s < ms) ? 1 : 0;
            eq += s == ms ? 1 : 0;
        }
    }
    for (int o = 1; o < (1 << shift); o <<= 1) {
        before += __shfl_xor_sync(0xffffffffu, before, o);
        eq += __shfl_xor_sync(0xffffffffu, eq, o);
    }
    if (active && sub == 0 && eq > self_in) {
        for (int j = 0; j < n; j++) {
            const Cand o = arr[j];
            if (o.score == ms && (o.label < me.label || (o.label == me.label && o.row < me.row))) before++;
        }
    }
    return before;
}

__device__ bool select_lists(const Cand *__restrict__ lists, int n_lists, int kp, FinSmem &sm, int tid) {
    Cand *S = sm.s;
    Cand *surv = S + kSelSurvCap;                                   // [kSelSurvCap]
    float *probe = reinterpret_cast<float *>(S + 2 * kSelSurvCap);  // [kSelProbeMax]
    const int m = (kp + n_lists - 1) / n_lists;
    const int n_probe = n_lists * m;
    if (tid < n_probe) probe[tid] = lists[(size_t)(tid / m) * kp + (tid % m)].score;
    if (tid == 0) sm.n_surv = 0u;
    __syncthreads();
    FIN_TRACE(1);
    {   // kp-th best probe (ties by index so that exactly one probe has that rank)
        const int shift = n_probe <= kFinThreads / 4 ? 2 : 1;
        const int ent = tid >> shift, sub = tid & ((1 << shift) - 1);
        const bool active = ent < n_probe;
        const float mine = active ? probe[ent] : 0.0f;
        int rank = 0;
        if (active) {
#pragma unroll 8
            for (int j = sub; j < n_probe; j += 1 << shift) {
                const float o = probe[j];
                rank += (o > mine || (o == mine && j < ent)) ? 1 : 0;
            }
        }
        for (int o = 1; o < (1 << shift); o <<= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
        if (active && sub == 0 && rank == kp - 1) sm.bound = mine;
    }
    __syncthreads();
    FIN_TRACE(2);
    const float lb = sm.bound;
    const int total = n_lists * kp;
#pragma unroll 4
    for (int i = tid; i < total; i += kFinThreads) {
        const Cand c = lists[i];
        if (c.row != kNoRow && c.score >= lb) {
            const uint32_t slot = atomicAdd(&sm.n_surv, 1u);
            if (slot < (uint32_t)kSelSurvCap) surv[slot] = c;
        }
    }
    __syncthreads();
    FIN_TRACE(3);
    const int n_surv = (int)sm.n_surv;
    if (n_surv > kSelSurvCap) return false;
    {
        const int shift = n_surv <= kFinThreads / 4 ? 2 : n_surv <= kFinThreads / 2 ? 1 : 0;
        const int ent = tid >> shift, sub = tid & ((1 << shift) - 1);
        const bool active = ent < n_surv;
        Cand me = empty_cand();
        if (active) me = surv[ent];
        const int rank = count_before<true>(surv, n_surv, me, active, sub, shift, 1);
        if (active && sub == 0 && rank < kp) S[rank] = me;
        if (tid >= n_surv && tid < kp) S[tid] = empty_cand();  // fewer than kp valid candidates in all lists together
    }
    return true;
}

__global__ void __launch_bounds__(kFinThreads, 1)
finalize_kernel(const __half *__restrict__ corpus, const float *__restrict__ queries,
                const Cand *__restrict__ partials, int n_lists, int kp, int k, float eps,
                uint64_t *__restrict__ labels_out, float *__restrict__ distances_out,
                uint32_t *__restrict__ counts_out, uint32_t *__restrict__ flags_out,
                const float *__restrict__ eps_q, const uint32_t *__restrict__ overflow, int scalar,
                uint32_t *__restrict__ counters, int n_counters, uint32_t *__restrict__ status_out, float eps_scale,
                uint32_t *__restrict__ stats, const float *__restrict__ corpus32) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    FinSmem &sm = *reinterpret_cast<FinSmem *>(smem_raw);
    const int tid = threadIdx.x;
    const int qi = blockIdx.x;
    const Cand *lists = partials + (size_t)qi * n_lists * kp;

    const int nthr = blockDim.x;
    FIN_TRACE(0);
    for (int c = tid; c < kDim; c += nthr) sm.q[c] = queries[(size_t)qi * kDim + c];

    // ---- K5: streaming tree merge, cap_lists lists per round, list 0 is the running result
    if (n_lists == 1) {  // already one sorted list (tensor-core path): nothing to merge
        for (int i = tid; i < kp; i += nthr) sm.s[i] = lists[i];
    } else if (n_lists * ((kp + n_lists - 1) / n_lists) <= kSelProbeMax && select_lists(lists, n_lists, kp, sm, tid)) {
        // sorted result already in sm.s[0..kp)
    } else {             // requires blockDim.x == kFinThreads
        __syncthreads();
        const int cap_lists = kFinCapEntries / kp;
        int next = 0;
        bool first = true;
        while (next < n_lists || first) {
            const int keep = first ? 0 : 1;
            const int take = min(cap_lists - keep, n_lists - next);
            for (int i = tid; i < take * kp; i += kFinThreads)
                sm.s[keep * kp + i] = lists[(size_t)next * kp + i];
            __syncthreads();
            merge_lists(sm.s, keep + take, kp, tid);
            next += take;
            first = false;
        }
    }
    __syncthreads();
    FIN_TRACE(4);

    // ---- K6: exact re-score.  The survivors' rows are first staged in shared memory by the whole CTA
    // (coalesced, one round trip to L2/HBM), then one thread per candidate adds the 384 products
    // sequentially in f32 -- the reference's order (vector.rs:128-134).
    // f32 rows (1536 B each) are read in place.  A single pre-merged list is read in place too: staging its k' = 128 rows was
    // measured slower (171 vs 127 us per 1024 queries; 100 KB of shared memory per CTA costs more occupancy than it saves).
    const bool stage_rows = n_lists > 1 && scalar != 2;
    const int entries = n_lists == 1 ? kp : kFinCapEntries;
    uint8_t *rows_sm = reinterpret_cast<uint8_t *>(sm.s + entries);
    const int stride = scalar ? kRowStrideI8 : kRowStrideF16;
    const int units = (scalar ? kDim : kRowBytesF16) / 16;  // 16-byte pieces per row
    for (int i = tid; stage_rows && i < kp * units; i += nthr) {
        const int c = i / units, j = i % units;
        const uint32_t row = sm.s[c].row;
        if (row != kNoRow) {
            const uint8_t *src = scalar ? reinterpret_cast<const uint8_t *>(corpus) + i8_row_offset(row)
                                        : reinterpret_cast<const uint8_t *>(corpus + (size_t)row * kDim);
            *reinterpret_cast<uint4 *>(rows_sm + c * stride + j * 16) = __ldg(reinterpret_cast<const uint4 *>(src) + j);
        }
    }
    __syncthreads();
    FIN_TRACE(5);
    Cand mine = empty_cand();
    float my_scan = __int_as_float(0x7f800000);  // scan score of this candidate (+inf for an empty slot)
    bool dropped = false;                        // a candidate whose exact score is NaN: not a result, yet it held a slot
    if (tid < kp) {
        mine = sm.s[tid];
        my_scan = mine.row != kNoRow ? mine.score : __int_as_float(0x7f800000);
        if (mine.row != kNoRow) {
            float acc = 0.0f;
            const uint4 *rp = stage_rows
                                  ? reinterpret_cast<const uint4 *>(rows_sm + tid * stride)
                                  : reinterpret_cast<const uint4 *>(
                                        scalar ? reinterpret_cast<const uint8_t *>(corpus) + i8_row_offset(mine.row)
                                               : reinterpret_cast<const uint8_t *>(corpus + (size_t)mine.row * kDim));
            if (scalar == 2) {
                // DAWN_SCALAR_F32: the exact score is over the f32 vector as it was added -- what the reference's
                // ScalarKind::F32 index stores (search_provider.rs:38) -- in the reference's order (vector.rs:128-134)
                const float4 *xp = reinterpret_cast<const float4 *>(corpus32 + (size_t)mine.row * kDim);
#pragma unroll 4
                for (int c = 0; c < kDim / 4; c++) {
                    const float4 x = __ldg(xp + c);
                    acc = __fadd_rn(acc, __fmul_rn(sm.q[4 * c], x.x));
                    acc = __fadd_rn(acc, __fmul_rn(sm.q[4 * c + 1], x.y));
                    acc = __fadd_rn(acc, __fmul_rn(sm.q[4 * c + 2], x.z));
                    acc = __fadd_rn(acc, __fmul_rn(sm.q[4 * c + 3], x.w));
                }
            } else if (scalar == 0) {
#pragma unroll 4
                for (int c = 0; c < kDim / 8; c++) {
                    const uint4 u = rp[c];
                    const __half2 *h = reinterpret_cast<const __half2 *>(&u);
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const float2 x = __half22float2(h[j]);
                        acc = __fadd_rn(acc, __fmul_rn(sm.q[c * 8 + 2 * j], x.x));
                        acc = __fadd_rn(acc, __fmul_rn(sm.q[c * 8 + 2 * j + 1], x.y));
                    }
                }
            } else {
                // int8 rows: score = scale * sum q[i]*f32(x[i]) (oracle/dawn_oracle.c:dawn_oracle_search_i8)
#pragma unroll 2
                for (int c = 0; c < kDim / 16; c++) {
                    const uint4 u = rp[c];
                    const int8_t *b8 = reinterpret_cast<const int8_t *>(&u);
#pragma unroll
                    for (int j = 0; j < 16; j++) acc = __fadd_rn(acc, __fmul_rn(sm.q[c * 16 + j], (float)b8[j]));
                }
                acc = __fmul_rn(*reinterpret_cast<const float *>(reinterpret_cast<const uint8_t *>(corpus) + i8_scale_offset(mine.row)), acc);
            }
            // evidence for the certificate's eps: the largest |selection score - exact score| ever seen (tests/test_gpu_slack.py)
            if (stats) {
                const float err = fabsf(my_scan - acc);
                if (err == err && __float_as_uint(err) > *reinterpret_cast<volatile uint32_t *>(&stats[2]))
                    atomicMax(&stats[2], __float_as_uint(err));
            }
            mine.score = __fsub_rn(1.0f, acc);  // distance, vector.rs:133
            if (acc != acc) {
                dropped = true;
                mine.row = kNoRow;
            }
        }
    }
    __syncthreads();  // every read of the merged list is done before it is overwritten with distances
    FIN_TRACE(6);
    // From here on Cand::score holds the DISTANCE (smaller is better); empty slots get +inf.
    const bool valid = tid < kp && mine.row != kNoRow;
    if (tid < kp) {
        if (mine.row == kNoRow) mine.score = __int_as_float(0x7f800000);
        sm.s[tid] = mine;
    }
    if (tid < kMaxCand) {  // weakest scan score among the candidates, one value per warp
        const uint32_t w = __reduce_min_sync(0xffffffffu, float_to_ordered(my_scan));
        if ((tid & 31) == 0) sm.warp_min[tid >> 5] = w;
    }
    if (tid < 32) {  // |q|^2: every eps below is proportional to |q| |x|
        float a = 0.f;
#pragma unroll
        for (int j = 0; j < kDim / 32; j++) a = fmaf(sm.q[tid + 32 * j], sm.q[tid + 32 * j], a);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
        if (tid == 0) sm.q_norm2 = a;
    }
    const int n_valid = __syncthreads_count(valid ? 1 : 0);
    const int n_held = __syncthreads_count(valid || dropped ? 1 : 0);  // candidates the lists held

    // ---- final order: distance asc, label asc, row asc (rank counting over <= 128 entries).
    // Ordering on the emitted f32 distance (not the score) makes the output self-consistent
    // and lets sharded results be merged from (label, distance) pairs alone.
    if (tid < kMaxCand) {
        const int rank = count_before<false>(sm.s, kp, mine, valid, 0, 0, 1);
        if (valid && rank < k) {
            labels_out[(size_t)qi * k + rank] = mine.label;
            distances_out[(size_t)qi * k + rank] = mine.score;
            if (rank == k - 1) sm.kth_dist = mine.score;
        }
    }
    __syncthreads();
    if (tid == 0) {
        counts_out[qi] = (uint32_t)min(k, n_valid);
        bool certified = true;
        if (n_held == kp) {
            // A row outside the candidate set has scan score <= scan_min, hence exact score
            // <= scan_min + eps and distance >= 1 - (scan_min + eps); it cannot displace or tie
            // the k-th result if that bound is strictly above the k-th distance.
            // the eps constants assume |q|, |x| inside the reference's gate (< 1.01); longer vectors scale them
            const float qn = sqrtf(sm.q_norm2);
            const float e = (eps_q ? eps_q[qi] : eps) * eps_scale * (qn > 1.01f ? qn * (1.001f / 1.01f) : 1.0f);
            uint32_t wmin = sm.warp_min[0];
            for (int w = 1; w < (kp + 31) / 32; w++) wmin = min(wmin, sm.warp_min[w]);
            const float scan_min = ordered_to_float(wmin);  // weakest kept candidate (lists need not be sorted)
            const float bound = __fsub_rn(1.0f, __fadd_rn(scan_min, e));
            certified = n_valid >= k && bound > sm.kth_dist;  // NaN drops can leave fewer than k: rows outside may be missing
        }
        if (overflow && overflow[qi]) certified = false;  // candidates were lost: cannot certify
        flags_out[qi] = certified ? 1u : 0u;
        if (!certified && stats) atomicAdd(&stats[0], 1u);
    }
    FIN_TRACE(7);
    // the last kernel of a search leaves the chunk counters / status word clean for the next one
    if (blockIdx.x == 0 && counters) {
        if (tid == 0 && status_out) *status_out = counters[0];
        if (tid == 0 && stats && counters[0]) atomicOr(&stats[1], counters[0]);
        __syncthreads();
        for (int i = tid; i < n_counters; i += nthr) counters[i] = 0u;
    }
    FIN_TRACE(8);
}

}  // namespace

namespace {
// see launch_score_error in dawn_common.cuh
__global__ void __launch_bounds__(256) score_error_kernel(const uint2 *__restrict__ log, const uint32_t *__restrict__ cnt,
                                                          int n_queries, int log_cap, const __half *__restrict__ corpus,
                                                          const float *__restrict__ q32, const __half *__restrict__ q16,
                                                          const float *__restrict__ eps_q, unsigned long long *__restrict__ out) {
    const int q = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double d_acc = 0.0, d_seq = 0.0, d_tot = 0.0, ratio = 0.0;
    bool have = false;
    if (q < n_queries && i < (int)min(cnt[q], (uint32_t)log_cap)) {
        const uint2 e = log[(size_t)q * log_cap + i];
        const float gemm = __uint_as_float(e.x);
        const __half *x = corpus + (size_t)e.y * kDim;
        const float *qf = q32 + (size_t)q * kDim;
        const __half *qh = q16 + (size_t)q * kDim;
        double dot16 = 0.0, dot32 = 0.0;
        float seq = 0.0f;
        for (int c = 0; c < kDim; c++) {
            const float xv = __half2float(x[c]);
            dot16 += (double)__half2float(qh[c]) * (double)xv;
            dot32 += (double)qf[c] * (double)xv;
            seq = __fadd_rn(seq, __fmul_rn(qf[c], xv));
        }
        d_acc = fabs((double)gemm - dot16);
        d_seq = fabs((double)seq - dot32);
        d_tot = fabs((double)gemm - (double)seq);
        ratio = d_tot / (double)eps_q[q];
        have = true;
        int ex;
        frexp(d_tot, &ex);  // d_tot in [2^(ex-1), 2^ex)
        int bin = d_tot == 0.0 ? 0 : ex + 39;  // bin b >= 1: [2^(b-40), 2^(b-39))
        bin = bin < 1 ? (d_tot == 0.0 ? 0 : 1) : (bin > 39 ? 39 : bin);
        atomicAdd(&out[8 + bin], 1ull);
    }
    // block maxima (doubles are non-negative: their bit patterns order like the values)
    __shared__ unsigned long long red[4][8];
    unsigned long long v[4] = {(unsigned long long)__double_as_longlong(d_acc), (unsigned long long)__double_as_longlong(d_seq),
                               (unsigned long long)__double_as_longlong(d_tot), (unsigned long long)__double_as_longlong(ratio)};
    const unsigned ballot = __ballot_sync(0xffffffffu, have);
    for (int k = 0; k < 4; k++) {
        for (int off = 16; off > 0; off >>= 1) {
            const unsigned long long o = __shfl_xor_sync(0xffffffffu, v[k], off);
            v[k] = o > v[k] ? o : v[k];
        }
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v[k];
    }
    __shared__ unsigned int s_pairs;
    if (threadIdx.x == 0) s_pairs = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) atomicAdd(&s_pairs, __popc(ballot));
    __syncthreads();
    if (threadIdx.x < 4) {
        unsigned long long m = 0;
        for (int w = 0; w < 8; w++) m = red[threadIdx.x][w] > m ? red[threadIdx.x][w] : m;
        atomicMax(&out[threadIdx.x], m);
    }
    if (threadIdx.x == 0) atomicAdd(&out[4], (unsigned long long)s_pairs);
}
}  // namespace

cudaError_t launch_score_error(const uint2 *log, const uint32_t *cnt, int n_queries, int log_cap, const __half *corpus,
                               const float *q32, const __half *q16, const float *eps_q, unsigned long long *out,
                               cudaStream_t s) {
    if (n_queries <= 0) return cudaSuccess;
    dim3 grid((unsigned)((log_cap + 255) / 256), (unsigned)n_queries);
    score_error_kernel<<<grid, 256, 0, s>>>(log, cnt, n_queries, log_cap, corpus, q32, q16, eps_q, out);
    return cudaGetLastError();
}

cudaError_t launch_finalize(const FinalizeLaunch &p, cudaStream_t s) {
    if (p.nq == 0) return cudaSuccess;
    if (p.kprime < 1 || p.kprime > kMaxCand || p.k < 1 || p.k > p.kprime) return cudaErrorInvalidValue;
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (p.scalar == 2 && !p.corpus32) return cudaErrorInvalidValue;
    const size_t smem = fin_smem_bytes(p.n_lists == 1 ? p.kprime : kFinCapEntries, p.kprime, p.scalar == 1 ? 1 : 0,
                                       p.n_lists > 1 && p.scalar != 2);
    if (dev < 64 && !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)fin_smem_bytes(kFinCapEntries, kMaxCand, 0, true));
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    finalize_kernel<<<p.nq, p.n_lists == 1 ? kFinThreadsSingle : kFinThreads, smem, s>>>(
        p.corpus, p.queries, p.partials, p.n_lists, p.kprime, p.k, p.eps, p.labels_out, p.distances_out, p.counts_out,
        p.flags_out, p.eps_q, p.overflow, p.scalar, p.counters, p.n_counters, p.status_out,
        p.eps_scale > 0.f ? p.eps_scale : 1.0f, p.stats, p.corpus32);
    return cudaGetLastError();
}

}  // namespace dawn
