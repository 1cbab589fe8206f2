// gemm_i8.cu -- K4c: large batches over an int8-stored corpus on the INT8 tensor cores
// (tcgen05.mma kind::i8, s32 accumulators in TMEM), straight from the blocked int8 arena: no dequantisation pass,
// no scratch.  Replaces usearch's Index::search (/root/reference/src/search/search_provider.rs:214) for batches over
// ScalarKind::F8-style storage (precedent: examples_old/search_usearch.rs:38, distance_i8 at src/search/vector.rs:157-163).
//
// Roofline: int8 tensor pipe for batch >~ 256 (2*B*N*384 int8 op), HBM below (388 B per row per pass) -- and, between the
// two, the TMEM READ port: a 128 x 256 s32 accumulator is 128 KB, tcgen05.ld moves 64 B/cycle/SM (B300_MICROARCH.md), i.e.
// 2048 cycles per tile, while the 12 MMAs of a tile (K = 384) take 1536 cycles at the int8 rate.  With K this short every
// accumulator element has to be read once, so the kernel cannot keep the int8 pipe more than 1536/2048 = 75 % busy; ncu shows
// 71 % (profiles/r02_gemm_i8_*).  (The fp16 kernel's tile takes 3072 MMA cycles for the same 2048 read cycles: tensor-bound.)
//
// How exactness survives an 8-bit query.  The MMA computes HI = sum_i hi_i * x8_i with ONE int8 level of the query
// (q ~ s1 * hi, |q - s1 hi|_2 =: delta ~ 8e-3), i.e. an approximate score a = s1 * s_row * HI with
// |a - exact| <= e1 = 1.03 * delta + 3e-6 (Cauchy-Schwarz; dequantised rows have norm < 1.02; the integer dot product
// itself is exact).  That is too loose to certify a top-k from approximate scores, so approximate scores are never
// ranked.  Instead:
//   * the epilogue only FILTERS: a row is appended to the query's candidate log iff a >= thr;
//   * select_i8_kernel re-scores every NEW log entry EXACTLY (the oracle's sequential f32 sum over the int8 row, times
//     the row scale: oracle/dawn_oracle.c:dawn_oracle_search_i8), keeps the best k' by exact score and publishes
//     thr = (k'-th best EXACT score) - e1 for the next round.
// A row the filter drops has a < T - e1, hence exact < T, hence it is not among the k' best: after the last round the
// log holds exactly the k' best rows of the whole corpus by exact score, whatever the distribution of the data.  The
// price of the one-level query is only a wider filter band (~2x more survivors on the synthetic corpus), not slack in
// the answer.  finalize.cu then orders them and emits 1 - score; its certificate sees exact scores (eps = 0).
// A log overflow (more than 2048 survivors in a round: massive near-ties) flags the query; the host API re-runs it
// through the exact scan, as on the fp16 path.
//
// Shape of one CTA (384 threads, 1 CTA/SM, persistent over work units):
//   A operand  = one 128-query tile of hi (int8), K-major, resident in shared memory: 3 k-blocks of 128 rows x 128 B  48 KB
//   B operand  = corpus tiles of 256 rows = 32 arena blocks, streamed k-block by k-block (256 x 128 B = 32 KB per stage)
//                by a 3-D TMA tensor map over the blocked arena {384 B row, 8 rows per block, blocks of 3104 B}   128 KB ring
//   scales     = the tile's 256 per-row f32 scales (they sit behind each block's rows), their own 2-D TMA map      8 x 1 KB ring
//   D          = 128 x 256 s32 in TMEM, two buffers; 12 MMAs (K = 32) per tile
//   warp 0 TMA producer, warp 1 MMA issuer + TMEM alloc, warps 4-11 epilogue: two warps per TMEM lane quarter, each
//   taking half of the tile's columns: tcgen05.ld -> I2F -> * scale -> max tree -> compare with the query's threshold.
//   CTA pairs (cta_group::2, M = 256) as in gemm_topk.cu when there is more than one query tile.
#include <cuda.h>

#include <cmath>

#include "dawn_common.cuh"
#include "gemm_pipe.cuh"

namespace dawn {

namespace {

using namespace pipe;

constexpr int kI8Threads = 384;
constexpr int BM = 128;             // queries per tile (UMMA M)
constexpr int BN = 256;             // corpus rows per tile (UMMA N) = 32 arena blocks
constexpr int BKB = 128;            // int8 elements (= bytes) per k-block = one swizzle-atom row
constexpr int kKBlocks = kDim / BKB;  // 3
constexpr int kUmmaKBytes = 32;     // one kind::i8 MMA covers K = 32
constexpr int kRingTiles32K = 4;    // B ring depth in 32 KB units: one int8 tile lasts ~1 us, about a DRAM round trip, so the ring
                                    // holds 1 1/3 tiles (the fp16 kernel's 3 stages hold half of its 2 us tile)
constexpr int kMaxStagesB = 2 * kRingTiles32K;  // 4 x 32 KB (one CTA) or 8 x 16 KB (CTA pair)
constexpr int kBRingBytes = kRingTiles32K * BN * BKB;  // 131072 either way
constexpr int kABlockBytes = BM * BKB;         // 16384
constexpr int kABytes = kABlockBytes * kKBlocks;  // 49152
constexpr int kTmemCols = 512;
constexpr int kEpiWarps = 8;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kStageCap = 16;       // survivors an epilogue thread parks in shared memory before one atomic flush
constexpr int kStagingBytes = kStageCap * kEpiThreads * 8;  // 32 KB
constexpr int kScaleSlots = 8;      // scale tiles in flight; the producer runs at most 5 tiles ahead of the epilogue
constexpr int kScaleTileBytes = BN * 4;
constexpr int kBarBytes = 512;
constexpr int kGroupMaxBytes = kEpiWarps * 32 * 4;  // per epilogue warp: the largest scale of each group of 4 columns
constexpr int kSmemBytes = 1024 + kABytes + kBRingBytes + kBarBytes + kScaleSlots * kScaleTileBytes + kStagingBytes + kGroupMaxBytes;

// Instruction descriptor for kind::i8: D = s32 (c_format 2 at bit 4), A = B = signed int8 (format 1 at bits 7 and 10),
// both K-major, N >> 3 at bit 17, M >> 4 at bit 24.
__host__ __device__ constexpr uint32_t make_idesc_i8(int m) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

struct I8Smem {  // offsets from the 1024-aligned base
    static constexpr int a_off = 0;
    static constexpr int b_off = kABytes;
    static constexpr int bar_off = kABytes + kBRingBytes;
    static constexpr int scale_off = bar_off + kBarBytes;
    static constexpr int staging_off = scale_off + kScaleSlots * kScaleTileBytes;
    static constexpr int groupmax_off = staging_off + kStagingBytes;
    // barriers (8 B each): full[6], empty[6], tmem_full[2], tmem_empty[2], a_full, a_free, scale_full[8]; then tmem ptr
};

#ifdef DAWN_COUNT_SLOW_PATH
// Measurement build only (make EXTRA=-DDAWN_COUNT_SLOW_PATH; tools/slow_path_count.py reads it): per launch of
// gemm_i8_topk_kernel, the epilogue's warp-chunks (32 queries x 32 columns) that went on to levels 2 and 3 (examine())
// and all warp-chunks processed.  slow_path_log_kernel, enqueued after each launch, moves the sums into a log.
__device__ unsigned long long g_slow_acc[2];
constexpr int kSlowLogCap = 4096;
__device__ unsigned long long g_slow_log[kSlowLogCap][4];  // {slow warp-chunks, warp-chunks, tiles of the launch, queries}
__device__ unsigned int g_slow_log_n;
__global__ void slow_path_log_kernel(uint32_t tiles, int n_queries) {
    const unsigned int i = g_slow_log_n;
    if (i < (unsigned int)kSlowLogCap) {
        g_slow_log[i][0] = g_slow_acc[0];
        g_slow_log[i][1] = g_slow_acc[1];
        g_slow_log[i][2] = tiles;
        g_slow_log[i][3] = (unsigned long long)n_queries;
        g_slow_log_n = i + 1;
    }
    g_slow_acc[0] = g_slow_acc[1] = 0ull;
}
#endif

__device__ __noinline__ void flush_staged_i8(uint32_t stage_smem, int col, uint32_t n, uint2 *__restrict__ log_q,
                                             uint32_t *__restrict__ cnt_q, uint32_t *__restrict__ overflow_q, int cap) {
    uint32_t slot = atomicAdd(cnt_q, n);
    for (uint32_t e = 0; e < n; e++, slot++) {
        uint2 val;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(val.x), "=r"(val.y) : "r"(stage_smem + (e * kEpiThreads + col) * 8));
        if (slot < (uint32_t)cap) log_q[slot] = val;
        else *overflow_q = 1u;
    }
}

template <int CG>
__global__ void __launch_bounds__(kI8Threads, 1)
gemm_i8_topk_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                    const __grid_constant__ CUtensorMap tmap_s, uint32_t tile_begin, uint32_t tile_end, uint32_t n_rows,
                    uint32_t n_tiles_total, uint32_t perm_mult, int n_qtiles, int n_queries, int chunk_tiles,
                    const float *__restrict__ thr_g, uint32_t *__restrict__ cnt_g, uint2 *__restrict__ log_g,
                    uint32_t *__restrict__ overflow_g, int log_cap, uint32_t *__restrict__ chunk_arrive,
                    const float *__restrict__ cq_g) {
    constexpr int kStagesB = kRingTiles32K * CG;
    constexpr int kBRows = BN / CG;                  // corpus rows this CTA streams per tile
    constexpr int kBStageBytes = kBRows * BKB;       // 32 KB or 16 KB
    constexpr uint32_t kIdesc = make_idesc_i8(BM * CG);
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t a_smem = base + I8Smem::a_off;
    const uint32_t b_smem = base + I8Smem::b_off;
    const uint32_t bars = base + I8Smem::bar_off;
    const uint32_t scale_smem = base + I8Smem::scale_off;
    auto full_bar = [&](int s) { return bars + 8 * s; };
    auto empty_bar = [&](int s) { return bars + 8 * (kMaxStagesB + s); };
    auto tfull_bar = [&](int a) { return bars + 8 * (2 * kMaxStagesB + a); };
    auto tempty_bar = [&](int a) { return bars + 8 * (2 * kMaxStagesB + 2 + a); };
    const uint32_t a_full_bar = bars + 8 * (2 * kMaxStagesB + 4);
    const uint32_t a_free_bar = bars + 8 * (2 * kMaxStagesB + 5);
    auto sfull_bar = [&](int s) { return bars + 8 * (2 * kMaxStagesB + 6 + s); };
    const uint32_t tmem_ptr_smem = bars + 8 * (2 * kMaxStagesB + 6 + kScaleSlots);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;  // 0 = leader (issues the MMAs)
    const uint32_t unit_first = blockIdx.x / CG;
    const uint32_t unit_stride = gridDim.x / CG;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStagesB; s++) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
        }
        for (int a = 0; a < 2; a++) {
            mbar_init(tfull_bar(a), 1);
            mbar_init(tempty_bar(a), kEpiWarps * CG);  // one arrival per epilogue warp (of both CTAs)
        }
        mbar_init(a_full_bar, 1);
        mbar_init(a_free_bar, 1);
        for (int s = 0; s < kScaleSlots; s++) mbar_init(sfull_bar(s), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        if constexpr (CG == 2) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_smem),
                         "r"((uint32_t)kTmemCols));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_smem),
                         "r"((uint32_t)kTmemCols));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
        }
    }
    tc_fence_before();
    if constexpr (CG == 2) cluster_sync_all();
    else __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_ptr_smem));

    // Work units and the strided visiting permutation: as in gemm_topk.cu.
    // (the 64-bit modulo is taken once per work unit; inside a unit the physical tile advances by perm_mult mod total)
    const uint32_t n_tiles = tile_end - tile_begin;
    auto phys_tile = [&](uint32_t tile) { return (uint32_t)(((uint64_t)(tile_begin + tile) * perm_mult) % n_tiles_total); };
    auto phys_next = [&](uint32_t pt) {
        const uint32_t nx = pt + perm_mult;  // perm_mult < n_tiles_total <= 2^24: no overflow
        return nx >= n_tiles_total ? nx - n_tiles_total : nx;
    };
    const uint32_t n_chunks = (n_tiles + chunk_tiles - 1) / chunk_tiles;
    const uint32_t n_units = n_chunks * (uint32_t)n_qtiles;

    if (warp == 0 && lane == 0) {
        // ===================== TMA producer (both CTAs of a pair) =====================
        uint32_t g = 0, n_reload = 0, tile_ctr = 0;
        int cur_t = -1;
        for (uint32_t u = unit_first; u < n_units; u += unit_stride) {
            const int t = (int)(u % (uint32_t)n_qtiles);
            const uint32_t chunk = u / (uint32_t)n_qtiles;
            if (t != cur_t) {
                if (n_reload > 0) mbar_wait(a_free_bar, (n_reload - 1) & 1u);
                const int qrow = t * BM * CG + (int)cta_rank * BM;
                if constexpr (CG == 2) {
                    if (cta_rank == 0) mbar_expect_tx(a_full_bar, 2 * kABytes);
                    const uint32_t lead = mapa_rank(a_full_bar, 0);
                    for (int kb = 0; kb < kKBlocks; kb++)
                        tma_load_2d_pair(a_smem + kb * kABlockBytes, &tmap_q, kb * BKB, qrow, lead);
                } else {
                    mbar_expect_tx(a_full_bar, kABytes);
                    for (int kb = 0; kb < kKBlocks; kb++)
                        tma_load_2d(a_smem + kb * kABlockBytes, &tmap_q, kb * BKB, qrow, a_full_bar);
                }
                cur_t = t;
                n_reload++;
            }
            if (chunk_arrive != nullptr && chunk < (uint32_t)kArriveSlots)  // start the chunk together with its other query tiles
                chunk_rendezvous(chunk_arrive + chunk, (uint32_t)n_qtiles, cta_rank == 0);
            const uint32_t tile0 = chunk * chunk_tiles;
            const uint32_t tile1 = min(n_tiles, tile0 + chunk_tiles);
            uint32_t pt = phys_tile(tile0);
            for (uint32_t tile = tile0; tile < tile1; tile++, tile_ctr++, pt = phys_next(pt)) {
                const uint32_t prow0 = pt * (uint32_t)BN;
                // The whole tile's 256 scales for THIS CTA's epilogue (each CTA of a pair filters all 256 columns
                // for its own 128 queries).  The slot being overwritten belonged to the tile 8 back; the B ring and
                // the two accumulators keep this producer at most 4 tiles ahead of the epilogue, so it is free.
                {
                    const uint32_t sl = tile_ctr % kScaleSlots;
                    mbar_expect_tx(sfull_bar(sl), kScaleTileBytes);
                    tma_load_2d(scale_smem + sl * kScaleTileBytes, &tmap_s, 0, (int)(prow0 / kI8BlockRows), sfull_bar(sl));
                }
                const int blk0 = (int)((prow0 + cta_rank * kBRows) / kI8BlockRows);
                for (int kb = 0; kb < kKBlocks; kb++, g++) {
                    const uint32_t s = g % kStagesB;
                    mbar_wait(empty_bar(s), ((g / kStagesB) & 1u) ^ 1u);
                    if constexpr (CG == 2) {
                        if (cta_rank == 0) mbar_expect_tx(full_bar(s), 2 * kBStageBytes);
                        tma_load_3d_pair(b_smem + s * kBStageBytes, &tmap_x, kb * BKB, 0, blk0, mapa_rank(full_bar(s), 0));
                    } else {
                        mbar_expect_tx(full_bar(s), kBStageBytes);
                        tma_load_3d(b_smem + s * kBStageBytes, &tmap_x, kb * BKB, 0, blk0, full_bar(s));
                    }
                }
            }
        }
    } else if (warp == 1 && lane == 0 && cta_rank == 0) {
        // ===================== MMA issuer (leader CTA only) =====================
        uint32_t g = 0, tile_ctr = 0, a_loads = 0;
        int cur_t = -1;
        for (uint32_t u = unit_first; u < n_units; u += unit_stride) {
            const int t = (int)(u % (uint32_t)n_qtiles);
            const uint32_t chunk = u / (uint32_t)n_qtiles;
            if (t != cur_t) {
                mbar_wait(a_full_bar, a_loads & 1u);
                a_loads++;
                cur_t = t;
            }
            const uint32_t tile0 = chunk * chunk_tiles;
            const uint32_t tile1 = min(n_tiles, tile0 + chunk_tiles);
            for (uint32_t tile = tile0; tile < tile1; tile++, tile_ctr++) {
                const uint32_t acc = tile_ctr & 1u;
                mbar_wait(tempty_bar(acc), ((tile_ctr >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < kKBlocks; kb++, g++) {
                    const uint32_t s = g % kStagesB;
                    mbar_wait(full_bar(s), (g / kStagesB) & 1u);
                    tc_fence_after();
                    const uint64_t adesc = make_kmajor_sw128_desc(a_smem + kb * kABlockBytes);
                    const uint64_t bdesc = make_kmajor_sw128_desc(b_smem + s * kBStageBytes);
#pragma unroll
                    for (int k = 0; k < BKB / kUmmaKBytes; k++) {
                        // advance 32 bytes inside the swizzle atom: +2 in 16-byte units
                        if constexpr (CG == 2)
                            tc_mma_i8_pair(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), kIdesc,
                                           (uint32_t)((kb | k) != 0));
                        else
                            tc_mma_i8(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), kIdesc,
                                      (uint32_t)((kb | k) != 0));
                    }
                    if constexpr (CG == 2) tc_commit_pair(empty_bar(s));
                    else tc_commit(empty_bar(s));
                }
                if constexpr (CG == 2) tc_commit_pair(tfull_bar(acc));
                else tc_commit(tfull_bar(acc));
            }
            const uint32_t u_next = u + unit_stride;
            if (u_next < n_units && (int)(u_next % (uint32_t)n_qtiles) != t) {
                if constexpr (CG == 2) tc_commit_pair(a_free_bar);
                else tc_commit(a_free_bar);
            }
        }
    } else if (warp >= 4) {
        // ===================== epilogue: threshold filter =====================
        // The test per element is  s_row * HI >= thr  (thr in units of s_row * HI, one per query = per thread).  Doing that
        // for every element costs I2F + FMUL + FMNMX each -- the first ncu capture had the tensor pipe 42 % busy waiting for
        // this.  Instead the test is hierarchical on INTEGER maxima: for a set S of columns, max_S(HI) * max_S(s_row) >= thr is
        // implied by any element of S passing (thr > 0, scales > 0).  Level 1: a 32-column chunk (16 three-input integer
        // maxima + one compare); level 2, only in chunks that pass: its 8 groups of 4 columns; level 3, only in groups that
        // pass: the 4 elements, exactly.  Once the thresholds have tightened almost every chunk stops at level 1.
        const int quarter = warp & 3;          // TMEM lane quarter this warp may read
        const int half = (warp - 4) >> 2;      // which 128 of the tile's 256 columns this warp filters
        const int col = (warp - 4) * 32 + lane;  // this thread's column in the staging area
        const uint32_t stage_smem = base + I8Smem::staging_off;
        const uint32_t gmax_smem = base + I8Smem::groupmax_off + (uint32_t)(warp - 4) * 128u;
        uint32_t n_st = 0;
        uint32_t tile_ctr = 0;
#ifdef DAWN_COUNT_SLOW_PATH
        uint32_t n_slow = 0, n_wchunks = 0;
#endif
        const uint32_t tempty_lead0 = CG == 2 ? mapa_rank(tempty_bar(0), 0) : 0u;
        const uint32_t tempty_lead1 = CG == 2 ? mapa_rank(tempty_bar(1), 0) : 0u;
        for (uint32_t u = unit_first; u < n_units; u += unit_stride) {
            const int t = (int)(u % (uint32_t)n_qtiles);
            const uint32_t chunk = u / (uint32_t)n_qtiles;
            const int q = t * BM * CG + (int)cta_rank * BM + quarter * 32 + lane;
            const bool q_valid = q < n_queries;
            const float thr = q_valid ? thr_g[q] : __int_as_float(0x7f800000);  // in units of s_row * (HI + cq)
            // shadow mode (the int8 rows are a quantised copy of fp16 rows that hold the truth): the row's own quantisation
            // error is bounded by ||q|| * kappa * s_row, i.e. by an offset cq = ||q|| * kappa / s1 on HI; 0 for an int8 corpus
            const float cq = q_valid ? cq_g[q] : 0.0f;
            const bool thr_pos = thr > 0.0f;  // the chunk bound needs a positive threshold (round 0 starts at -inf)
            uint2 *log_q = log_g + (size_t)q * log_cap;
            const uint32_t tile0 = chunk * chunk_tiles;
            const uint32_t tile1 = min(n_tiles, tile0 + chunk_tiles);
            uint32_t pt = phys_tile(tile0);
            for (uint32_t tile = tile0; tile < tile1; tile++, tile_ctr++, pt = phys_next(pt)) {
                const uint32_t acc = tile_ctr & 1u;
                const uint32_t row0 = pt * (uint32_t)BN;
                const uint32_t sl = tile_ctr % kScaleSlots;
                const uint32_t sc_addr = scale_smem + sl * kScaleTileBytes + half * (BN / 2) * 4;
                mbar_wait(sfull_bar(sl), (tile_ctr / kScaleSlots) & 1u);
                // largest scale of each group of 4 columns (lane l: columns 4l..4l+3 of this half tile) -> this warp's
                // shared array, and of each 32-column chunk (8 lanes) -> register
                float smax;
                {
                    float4 s4;
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                                 : "=f"(s4.x), "=f"(s4.y), "=f"(s4.z), "=f"(s4.w)
                                 : "r"(sc_addr + (uint32_t)lane * 16u));
                    smax = fmaxf(fmaxf(s4.x, s4.y), fmaxf(s4.z, s4.w));
                    asm volatile("st.shared.f32 [%0], %1;" ::"r"(gmax_smem + (uint32_t)lane * 4u), "f"(smax) : "memory");
                    smax = fmaxf(smax, __shfl_xor_sync(0xffffffffu, smax, 1));
                    smax = fmaxf(smax, __shfl_xor_sync(0xffffffffu, smax, 2));
                    smax = fmaxf(smax, __shfl_xor_sync(0xffffffffu, smax, 4));  // every lane of group l/8 holds chunk l/8's max
                    __syncwarp();
                }
                mbar_wait(tfull_bar(acc), (tile_ctr >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN + half * (BN / 2);
                const int lim_tile = (int)n_rows - (int)row0 - half * (BN / 2);  // valid columns of this half tile
                // levels 2 and 3 for one chunk (rare once thresholds are tight)
                auto examine = [&](const uint32_t (&v)[32], const int (&m)[8], int c) {
                    float gs[8];
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                                 : "=f"(gs[0]), "=f"(gs[1]), "=f"(gs[2]), "=f"(gs[3])
                                 : "r"(gmax_smem + (uint32_t)c * 32u));
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                                 : "=f"(gs[4]), "=f"(gs[5]), "=f"(gs[6]), "=f"(gs[7])
                                 : "r"(gmax_smem + (uint32_t)c * 32u + 16u));
#pragma unroll
                    for (int g = 0; g < 8; g++) {
                        if (thr_pos && !((__int2float_rn(m[g]) + cq) * gs[g] >= thr)) continue;
                        float4 s4;
                        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                                     : "=f"(s4.x), "=f"(s4.y), "=f"(s4.z), "=f"(s4.w)
                                     : "r"(sc_addr + (uint32_t)(c * 32 + g * 4) * 4u));
                        const float sc[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const int i = 4 * g + j;
                            const float f = (__int2float_rn((int)v[i]) + cq) * sc[j];
                            if (f >= thr && c * 32 + i < lim_tile) {
                                asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(stage_smem + (n_st * kEpiThreads + col) * 8),
                                             "r"(__float_as_uint(f)), "r"(row0 + half * (BN / 2) + c * 32 + i)
                                             : "memory");
                                if (++n_st == (uint32_t)kStageCap) {
                                    flush_staged_i8(stage_smem, col, n_st, log_q, cnt_g + q, overflow_g + q, log_cap);
                                    n_st = 0;
                                }
                            }
                        }
                    }
                };
                auto process = [&](const uint32_t (&v)[32], int c) {
                    int m[8];
#pragma unroll
                    for (int g = 0; g < 8; g++)
                        m[g] = max(max((int)v[4 * g], (int)v[4 * g + 1]), max((int)v[4 * g + 2], (int)v[4 * g + 3]));
                    const int mm = max(max(max(m[0], m[1]), max(m[2], m[3])), max(max(m[4], m[5]), max(m[6], m[7])));
                    const float sm_c = __shfl_sync(0xffffffffu, smax, 8 * c);
                    const bool hit = q_valid && (!thr_pos || (__int2float_rn(mm) + cq) * sm_c >= thr);
#ifdef DAWN_COUNT_SLOW_PATH
                    n_slow += __any_sync(0xffffffffu, hit) ? 1u : 0u;
                    n_wchunks++;
#endif
                    if (hit) examine(v, m, c);
                    __syncwarp();
                };
                uint32_t v0[32], v1[32];
                tc_ld_32x32b_x32(taddr, v0);
#pragma unroll 1
                for (int c = 0; c < BN / 2 / 32; c += 2) {
                    tc_wait_ld();
                    tc_ld_32x32b_x32(taddr + (c + 1) * 32, v1);
                    process(v0, c);
                    tc_wait_ld();
                    if (c + 2 < BN / 2 / 32) tc_ld_32x32b_x32(taddr + (c + 2) * 32, v0);
                    process(v1, c + 1);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if constexpr (CG == 2) mbar_arrive_cluster(acc ? tempty_lead1 : tempty_lead0);
                    else mbar_arrive(tempty_bar(acc));
                }
                if (__any_sync(0xffffffffu, n_st >= (uint32_t)(kStageCap / 2))) {
                    if (n_st) flush_staged_i8(stage_smem, col, n_st, log_q, cnt_g + q, overflow_g + q, log_cap);
                    n_st = 0;
                    __syncwarp();
                }
            }
            if (n_st) {  // the next unit belongs to another query tile
                flush_staged_i8(stage_smem, col, n_st, log_q, cnt_g + q, overflow_g + q, log_cap);
                n_st = 0;
            }
            __syncwarp();
        }
#ifdef DAWN_COUNT_SLOW_PATH
        if (lane == 0) {
            atomicAdd(&g_slow_acc[0], (unsigned long long)n_slow);
            atomicAdd(&g_slow_acc[1], (unsigned long long)n_wchunks);
        }
#endif
    }

    tc_fence_before();
    if constexpr (CG == 2) cluster_sync_all();
    else __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        __syncwarp();
        if constexpr (CG == 2)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)kTmemCols));
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)kTmemCols));
    }
}

// ---- query preparation: f32 -> one int8 level hi (padded to whole tiles), s1, and the filter band e1 -----------
// kappa > 0 = shadow mode: the int8 rows are quantised copies (error norm <= kappa * s_row, measured when they were made) of
// fp16 rows that hold the truth; cq_g[q] = ||q|| * kappa / s1 is the offset the epilogue adds to HI, and e1 also covers the
// longer dequantised rows (norm <= 1.0105 + kappa * s_row <= 1.09) and the f32 rounding of the exact sequential sum.
__global__ void __launch_bounds__(128) prep_queries_i8_gemm_kernel(const float *__restrict__ q32, int n_queries,
                                                                   int8_t *__restrict__ q8, float *__restrict__ s1_g,
                                                                   float *__restrict__ e1_g, float *__restrict__ cq_g,
                                                                   float kappa) {
    const int q = blockIdx.x;
    __shared__ float red[4];
    __shared__ float red2[4];
    float x[3], amax = 0.f;
#pragma unroll
    for (int j = 0; j < 3; j++) {
        x[j] = q < n_queries ? q32[(size_t)q * kDim + threadIdx.x + 128 * j] : 0.f;
        amax = fmaxf(amax, fabsf(x[j]));
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, off));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = amax;
    __syncthreads();
    amax = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
    const float s1 = amax > 0.f ? amax / 127.0f : 1.0f;
    float err2 = 0.f, n2 = 0.f;
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const int hi = max(-127, min(127, (int)rintf(x[j] / s1)));
        const float e = fmaf(-s1, (float)hi, x[j]);
        err2 += e * e;
        n2 = fmaf(x[j], x[j], n2);
        q8[(size_t)q * kDim + threadIdx.x + 128 * j] = (int8_t)hi;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        err2 += __shfl_xor_sync(0xffffffffu, err2, off);
        n2 += __shfl_xor_sync(0xffffffffu, n2, off);
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) {
        red[threadIdx.x >> 5] = err2;
        red2[threadIdx.x >> 5] = n2;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        s1_g[q] = s1;
        const float delta = sqrtf(red[0] + red[1] + red[2] + red[3]);
        if (kappa > 0.0f) {
            // shadow mode: |q.x16 - s1 s_row HI| <= ||q - s1 hi|| * ||s_row x8|| + ||q|| * ||x16 - s_row x8||; the second term is
            // row-dependent and lives in cq; 3e-5 = the f32 rounding of the exact sequential sum (<= 384 * 2^-24 * 1.03) plus the
            // roundings of a and thr / s1
            e1_g[q] = delta * 1.10f + 3.0e-5f;
            cq_g[q] = sqrtf(red2[0] + red2[1] + red2[2] + red2[3]) * 1.00001f * kappa / s1;
        } else {
            // |sum (q_i - s1 hi_i) x_i| <= ||q - s1 hi|| * ||x||, dequantised rows have norm < 1.02; 1.03 also covers the f32
            // rounding of this sum of squares; + 3e-6 for the f32 roundings of a = s1 * (s_row * HI) and of thr / s1.
            e1_g[q] = delta * 1.03f + 3.0e-6f;
            cq_g[q] = 0.0f;
        }
    }
}

// ---- select: re-score the round's new log entries EXACTLY, keep the best k', publish the next threshold ----------
// Entries [0, kept_g[q]) of the log carry exact scores from the previous select; entries [kept, cnt) were appended by
// the round just finished and carry the filter's approximate value, which is ignored.  The exact score is the oracle's:
// scale * (sequential f32 sum of q[i] * f32(x8[i])), oracle/dawn_oracle.c:dawn_oracle_search_i8 -- the same arithmetic
// finalize.cu uses, so the final distances are bit-identical.
__global__ void __launch_bounds__(kSelThreads) select_i8_kernel(uint2 *__restrict__ log_g, uint32_t *__restrict__ cnt_g,
                                                                uint32_t *__restrict__ kept_g, float *__restrict__ thr_g,
                                                                uint32_t *__restrict__ overflow_g, int log_cap, int kp,
                                                                const uint8_t *__restrict__ arena,
                                                                const float *__restrict__ q32, int n_queries,
                                                                const float *__restrict__ s1_g, const float *__restrict__ e1_g,
                                                                float limit_score, float eps_scale,
                                                                const uint64_t *__restrict__ labels,
                                                                Cand *__restrict__ final_lists, uint32_t *__restrict__ arrive,
                                                                const __half *__restrict__ corpus16) {
    __shared__ unsigned long long keys[kSelCap];
    clear_arrive_slots(arrive, blockIdx.x, gridDim.x, threadIdx.x, kSelThreads);
    __shared__ unsigned long long s_prefix;
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s_need, s_out, s_marked;
    __shared__ float s_qn2;
    __shared__ __align__(16) float sq[kDim];
    __shared__ uint16_t s_list[kSelCap];  // new entries that need the exact re-score
    // rows of the entries being re-scored exactly, staged by the whole CTA: strides of 49 / 25 x 16 B keep the eight threads of a
    // quarter warp on different 16-byte bank groups
    constexpr int kPassRows = 24, kStride16 = 2 * kDim + 16, kStride8 = kDim + 16;
    __shared__ __align__(16) uint8_t s_rows[kPassRows * kStride16];
    __shared__ float s_scale[kPassRows];
    const int q = blockIdx.x;
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    uint2 *log_q = log_g + (size_t)q * log_cap;
    const uint32_t cnt = cnt_g[q];
    const int n = (int)min(cnt, (uint32_t)log_cap);
    const int kept = (int)min(kept_g[q], (uint32_t)n);
    for (int c = tid; c < kDim; c += kSelThreads) sq[c] = q < n_queries ? q32[(size_t)q * kDim + c] : 0.f;
    if (tid == 0) {
        s_prefix = 0ull;
        s_need = (uint32_t)kp;
        s_out = 0u;
        s_marked = 0u;
    }
    __syncthreads();
    // ---- stage A: a fast f32 score of every NEW entry, one warp per entry (coalesced row read, 12 elements per lane, fma +
    // shuffle tree).  It differs from the exact (sequential, unfused) score by at most eta: both are within
    // 384 * 2^-24 * |q| |x| of the real dot product.
    float ql[12];
#pragma unroll
    for (int j = 0; j < 12; j++) ql[j] = sq[12 * lane + j];
    if (warp == 0) {
        float a = 0.f;
#pragma unroll
        for (int j = 0; j < 12; j++) a = fmaf(ql[j], ql[j], a);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
        if (lane == 0) s_qn2 = a;
    }
    for (int i = tid; i < kept; i += kSelThreads) {  // exact scores from the previous select
        const uint2 e = log_q[i];
        keys[i] = ((unsigned long long)float_to_ordered(__uint_as_float(e.x)) << 32) | (unsigned long long)(~e.y);
    }
    // A handful of queries means a handful of CTAs on the whole GPU: the select is then pure latency, and one thread per
    // entry doing the exact re-score straight away (256 entries in flight per CTA, no second pass) is quicker than the
    // stages below (12.5M rows, one query: 0.97 against 1.10 ms per search).
    const bool one_stage = n_queries <= 64;
    for (int i = kept + tid; one_stage && i < n; i += kSelThreads) {
        const uint32_t row = log_q[i].y;
        float acc = 0.0f;
        if (corpus16) {
            const uint4 *rp = reinterpret_cast<const uint4 *>(corpus16 + (size_t)row * kDim);
#pragma unroll 4
            for (int c = 0; c < kDim / 8; c++) {
                const uint4 u = __ldg(rp + c);
                const __half2 *h = reinterpret_cast<const __half2 *>(&u);
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const float2 x = __half22float2(h[j]);
                    acc = __fadd_rn(acc, __fmul_rn(sq[c * 8 + 2 * j], x.x));
                    acc = __fadd_rn(acc, __fmul_rn(sq[c * 8 + 2 * j + 1], x.y));
                }
            }
        } else {
            const uint4 *rp = reinterpret_cast<const uint4 *>(arena + i8_row_offset(row));
#pragma unroll 2
            for (int c = 0; c < kDim / 16; c++) {
                const uint4 u = __ldg(rp + c);
                const int8_t *b8 = reinterpret_cast<const int8_t *>(&u);
#pragma unroll
                for (int j = 0; j < 16; j++) acc = __fadd_rn(acc, __fmul_rn(sq[c * 16 + j], (float)b8[j]));
            }
            acc = __fmul_rn(*reinterpret_cast<const float *>(arena + i8_scale_offset(row)), acc);
        }
        keys[i] = ((unsigned long long)float_to_ordered(acc) << 32) | (unsigned long long)(~row);
    }
#pragma unroll 2
    for (int i = kept + warp; !one_stage && i < n; i += kSelThreads / 32) {
        const uint32_t row = log_q[i].y;
        float a = 0.f;
        if (corpus16) {
            const uint2 *src = reinterpret_cast<const uint2 *>(corpus16 + (size_t)row * kDim) + lane * 3;
            uint2 u[3];
#pragma unroll
            for (int j = 0; j < 3; j++) u[j] = __ldg(src + j);
#pragma unroll
            for (int j = 0; j < 3; j++) {
                const __half2 *h = reinterpret_cast<const __half2 *>(&u[j]);
                const float2 x0 = __half22float2(h[0]), x1 = __half22float2(h[1]);
                a = fmaf(ql[4 * j], x0.x, a);
                a = fmaf(ql[4 * j + 1], x0.y, a);
                a = fmaf(ql[4 * j + 2], x1.x, a);
                a = fmaf(ql[4 * j + 3], x1.y, a);
            }
        } else {
            const uint32_t *src = reinterpret_cast<const uint32_t *>(arena + i8_row_offset(row)) + lane * 3;
            uint32_t u[3];
#pragma unroll
            for (int j = 0; j < 3; j++) u[j] = __ldg(src + j);
#pragma unroll
            for (int j = 0; j < 3; j++) {
                const int8_t *b8 = reinterpret_cast<const int8_t *>(&u[j]);
#pragma unroll
                for (int e = 0; e < 4; e++) a = fmaf(ql[4 * j + e], (float)b8[e], a);
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
        if (!corpus16) a *= *reinterpret_cast<const float *>(arena + i8_scale_offset(row));
        if (lane == 0) keys[i] = ((unsigned long long)float_to_ordered(a) << 32) | (unsigned long long)(~row);
    }
    __syncthreads();
    // ---- stage B: tau = the k'-th best fast score.  At least k' entries then have an exact score >= tau - eta, so an entry
    // whose fast score is below tau - 2 eta (exact < tau - eta) is not among the k' best: only the others are re-scored exactly.
    float cut = __int_as_float(0xff800000);
    if (n >= kp && n > kept && !one_stage) {
        const unsigned long long Kt = radix_select_kth(keys, n, kp, hist, &s_prefix, &s_need, tid);
        const float eta = 6.0e-5f * fmaxf(1.0f, sqrtf(s_qn2)) * eps_scale;
        cut = ordered_to_float((uint32_t)(Kt >> 32)) - 2.0f * eta;
        __syncthreads();
        if (tid == 0) {
            s_prefix = 0ull;
            s_need = (uint32_t)kp;
        }
    }
    for (int i = kept + tid; !one_stage && i < n; i += kSelThreads) {
        if (ordered_to_float((uint32_t)(keys[i] >> 32)) >= cut) s_list[atomicAdd(&s_marked, 1u)] = (uint16_t)i;
        else keys[i] = (unsigned long long)i;  // dropped: below every real key (and distinct)
    }
    __syncthreads();
    // ---- stage C: the exact score (the oracle's sequential f32 sum) of the marked entries, rows staged through shared memory
    const int n_marked = (int)s_marked;
    const int units = corpus16 ? 2 * kDim / 16 : kDim / 16;  // 16-byte pieces per row
    const int stride = corpus16 ? kStride16 : kStride8;
    for (int base = 0; base < n_marked; base += kPassRows) {
        const int m = min(kPassRows, n_marked - base);
        for (int u = tid; u < m * units; u += kSelThreads) {
            const int r = u / units, j = u - r * units;
            const uint32_t row = ~(uint32_t)keys[s_list[base + r]];
            const uint8_t *src = corpus16 ? reinterpret_cast<const uint8_t *>(corpus16 + (size_t)row * kDim) : arena + i8_row_offset(row);
            *reinterpret_cast<uint4 *>(s_rows + r * stride + j * 16) = __ldg(reinterpret_cast<const uint4 *>(src) + j);
        }
        if (!corpus16 && tid < m)
            s_scale[tid] = *reinterpret_cast<const float *>(arena + i8_scale_offset(~(uint32_t)keys[s_list[base + tid]]));
        __syncthreads();
        if (tid < m) {
            const uint4 *rp = reinterpret_cast<const uint4 *>(s_rows + tid * stride);
            float acc = 0.0f;
            if (corpus16) {
#pragma unroll 4
                for (int c = 0; c < kDim / 8; c++) {
                    const uint4 u = rp[c];
                    const float4 qa = *reinterpret_cast<const float4 *>(&sq[c * 8]), qb = *reinterpret_cast<const float4 *>(&sq[c * 8 + 4]);
                    const __half2 *h = reinterpret_cast<const __half2 *>(&u);
                    const float2 x0 = __half22float2(h[0]), x1 = __half22float2(h[1]), x2 = __half22float2(h[2]), x3 = __half22float2(h[3]);
                    acc = __fadd_rn(acc, __fmul_rn(qa.x, x0.x));
                    acc = __fadd_rn(acc, __fmul_rn(qa.y, x0.y));
                    acc = __fadd_rn(acc, __fmul_rn(qa.z, x1.x));
                    acc = __fadd_rn(acc, __fmul_rn(qa.w, x1.y));
                    acc = __fadd_rn(acc, __fmul_rn(qb.x, x2.x));
                    acc = __fadd_rn(acc, __fmul_rn(qb.y, x2.y));
                    acc = __fadd_rn(acc, __fmul_rn(qb.z, x3.x));
                    acc = __fadd_rn(acc, __fmul_rn(qb.w, x3.y));
                }
            } else {
#pragma unroll 2
                for (int c = 0; c < kDim / 16; c++) {
                    const uint4 u = rp[c];
                    const int8_t *b8 = reinterpret_cast<const int8_t *>(&u);
#pragma unroll
                    for (int j = 0; j < 16; j++) acc = __fadd_rn(acc, __fmul_rn(sq[c * 16 + j], (float)b8[j]));
                }
                acc = __fmul_rn(s_scale[tid], acc);
            }
            const int i = s_list[base + tid];
            keys[i] = ((unsigned long long)float_to_ordered(acc) << 32) | (keys[i] & 0xffffffffull);
        }
        __syncthreads();
    }
    const unsigned long long K = n >= kp ? radix_select_kth(keys, n, kp, hist, &s_prefix, &s_need, tid) : 0ull;
    for (int i = tid; i < n; i += kSelThreads) {
        const unsigned long long key = keys[i];
        if (key >= K) {
            const uint32_t pos = atomicAdd(&s_out, 1u);
            if (pos < (uint32_t)kp) {
                const float sc = ordered_to_float((uint32_t)(key >> 32));
                const uint32_t row = ~(uint32_t)key;
                log_q[pos] = make_uint2(__float_as_uint(sc), row);
                if (final_lists) {
                    Cand c;
                    c.score = sc;
                    c.row = row;
                    c.label = labels[row];
                    final_lists[(size_t)q * kp + pos] = c;
                }
            }
        }
    }
    __syncthreads();
    const int keep = min(n, kp);
    if (final_lists)
        for (int i = keep + tid; i < kp; i += kSelThreads) final_lists[(size_t)q * kp + i] = empty_cand();
    if (tid == 0) {
        cnt_g[q] = (uint32_t)keep;
        kept_g[q] = (uint32_t)keep;
        float T = n >= kp ? ordered_to_float((uint32_t)(K >> 32)) : __int_as_float(0xff800000);
        // distance_limit pushed down: rows whose exact score is below limit_score are dropped by the caller anyway
        if (limit_score > __int_as_float(0xff800000)) T = fmaxf(T, limit_score - 1e-6f);
        // filter threshold in the epilogue's units (s_row * HI): a row with a < T - e1 has exact < T
        const float s1 = q < n_queries ? s1_g[q] : 1.0f;
        const float e1 = q < n_queries ? e1_g[q] * eps_scale : 0.f;
        thr_g[q] = T > __int_as_float(0xff800000) ? (T - e1) / s1 - fabsf((T - e1) / s1) * 4.0e-7f : T;
        if (cnt > (uint32_t)log_cap) overflow_g[q] = 1u;
    }
}

// Blocked int8 arena as a 3-D tensor {384 B of a row, 8 rows of a block, blocks 3104 B apart}; box = 128 B x 8 x box_blocks
// lands in shared memory as box_blocks*8 consecutive 128-byte rows = the canonical K-major SWIZZLE_128B operand layout.
bool make_tmap_arena(CUtensorMap *map, const void *arena, uint64_t n_blocks, uint32_t box_blocks) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return false;
    cuuint64_t dims[3] = {(cuuint64_t)kDim, (cuuint64_t)kI8BlockRows, (cuuint64_t)n_blocks};
    cuuint64_t strides[2] = {(cuuint64_t)kDim, (cuuint64_t)kI8BlockBytes};
    cuuint32_t box[3] = {(cuuint32_t)BKB, (cuuint32_t)kI8BlockRows, box_blocks};
    cuuint32_t estr[3] = {1, 1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void *>(arena), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// The 8 f32 scales behind each block's rows as a 2-D tensor {8 floats, blocks 3104 B apart}; box = 8 x 32 = one tile's 256 scales.
bool make_tmap_scales(CUtensorMap *map, const void *arena, uint64_t n_blocks) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)kI8BlockRows, (cuuint64_t)n_blocks};
    cuuint64_t strides[1] = {(cuuint64_t)kI8BlockBytes};
    cuuint32_t box[2] = {(cuuint32_t)kI8BlockRows, (cuuint32_t)(BN / kI8BlockRows)};
    cuuint32_t estr[2] = {1, 1};
    const uint8_t *base = static_cast<const uint8_t *>(arena) + (size_t)kI8BlockRows * kDim;
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<uint8_t *>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// hi queries [rows][384] int8 row-major, box = 128 B x 128 rows, 128 B swizzle
bool make_tmap_q8(CUtensorMap *map, const void *base, uint64_t rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)kDim, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)kDim};
    cuuint32_t box[2] = {(cuuint32_t)BKB, (cuuint32_t)BM};
    cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int CG>
cudaError_t launch_round(int grid, cudaStream_t s, const CUtensorMap &tq, const CUtensorMap &tx, const CUtensorMap &ts,
                         uint32_t tile_begin, uint32_t tile_end, uint32_t n_rows, uint32_t n_tiles_total, uint32_t perm_mult,
                         int n_qtiles, int n_queries, int chunk, const float *thr, uint32_t *cnt, uint2 *log,
                         uint32_t *overflow, uint32_t *arrive, const float *cq) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kI8Threads);
    cfg.dynamicSmemBytes = kSmemBytes;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int log_cap = kSelCap;
    return cudaLaunchKernelEx(&cfg, gemm_i8_topk_kernel<CG>, tq, tx, ts, tile_begin, tile_end, n_rows, n_tiles_total, perm_mult,
                              n_qtiles, n_queries, chunk, thr, cnt, log, overflow, log_cap, arrive, cq);
}

}  // namespace

size_t gemm_i8_workspace_bytes(int n_queries) {
    const size_t qp = ((size_t)n_queries + 2 * BM - 1) / (2 * BM) * (2 * BM);
    return qp * kDim + qp * (7 * sizeof(float)) + qp * (size_t)kSelCap * sizeof(uint2) + 1024 + kArriveSlots * sizeof(uint32_t);
}

cudaError_t launch_gemm_search_i8(const GemmSearchI8 &p, cudaStream_t s) {
    if (p.n_queries <= 0 || p.n_rows == 0) return cudaErrorInvalidValue;
    int cg = p.cta_group;
    if (cg != 1 && cg != 2) cg = p.n_queries > BM ? 2 : 1;
    if (p.grid % 2) cg = 1;
    const int qtile = BM * cg;
    const int qp = (p.n_queries + qtile - 1) / qtile * qtile;
    const int n_qtiles = qp / qtile;
    const int workers = p.grid / cg;
    uint8_t *w = static_cast<uint8_t *>(p.workspace);
    int8_t *q8 = reinterpret_cast<int8_t *>(w);
    w += (size_t)qp * kDim;
    float *s1 = reinterpret_cast<float *>(w);
    w += (size_t)qp * sizeof(float);
    float *e1 = reinterpret_cast<float *>(w);
    w += (size_t)qp * sizeof(float);
    float *thr = reinterpret_cast<float *>(w);
    w += (size_t)qp * sizeof(float);
    uint32_t *cnt = reinterpret_cast<uint32_t *>(w);
    w += (size_t)qp * sizeof(uint32_t);
    uint32_t *kept = reinterpret_cast<uint32_t *>(w);
    w += (size_t)qp * sizeof(uint32_t);
    uint32_t *overflow = reinterpret_cast<uint32_t *>(w);
    w += (size_t)qp * sizeof(uint32_t);
    float *cq = reinterpret_cast<float *>(w);
    w += (size_t)qp * sizeof(float);
    w = reinterpret_cast<uint8_t *>(((uintptr_t)w + 255) & ~(uintptr_t)255);
    uint2 *log = reinterpret_cast<uint2 *>(w);
    uint32_t *arrive = (n_qtiles > 1 && !p.no_unit_sync) ? reinterpret_cast<uint32_t *>(w + (size_t)qp * kSelCap * sizeof(uint2)) : nullptr;

    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 64 && !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(gemm_i8_topk_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(gemm_i8_topk_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    const uint64_t n_blocks = (p.n_rows + kI8BlockRows - 1) / kI8BlockRows;
    CUtensorMap tq, tx, ts;
    if (!make_tmap_q8(&tq, q8, (uint64_t)qp) || !make_tmap_arena(&tx, p.arena, n_blocks, (uint32_t)(BN / cg / kI8BlockRows)) ||
        !make_tmap_scales(&ts, p.arena, n_blocks))
        return cudaErrorInvalidValue;

    cudaError_t e;
    if ((e = cudaMemsetAsync(cnt, 0, (size_t)qp * 3 * sizeof(uint32_t), s)) != cudaSuccess) return e;  // cnt, kept, overflow
    const float kappa = p.rescore_f16 ? p.shadow_kappa : 0.0f;
    if (p.rescore_f16 && !(kappa > 0.0f)) return cudaErrorInvalidValue;
    prep_queries_i8_gemm_kernel<<<qp, 128, 0, s>>>(p.queries, p.n_queries, q8, s1, e1, cq, kappa);
    // thresholds before the first round: -inf, or the pushed-down limit (a select pass over empty logs)
    select_i8_kernel<<<qp, kSelThreads, 0, s>>>(log, cnt, kept, thr, overflow, kSelCap, p.kprime, p.arena, p.queries,
                                                p.n_queries, s1, e1, p.limit_score, p.eps_scale, p.labels, nullptr, arrive,
                                                p.rescore_f16);
    int launches = 2;
    // Rounds grow x8 (x4 for k' = 128): the filter band e1 lets ~2x more rows through than an exact threshold would,
    // (growth - 1) * k' * 2.2 + k' entries must fit the 2048-entry log with margin.
    // Shadow mode: the band also holds the rows' own quantisation error (~5x the survivors of an exact threshold).
    uint64_t growth = p.kprime > 64 ? 4 : 8;
    if (p.growth >= 2) growth = (uint64_t)p.growth;
    const uint64_t band_x4 = p.rescore_f16 ? 22 : 11;  // survivors per exact-threshold survivor, in quarters
    while (growth > 2 && (growth - 1) * (uint64_t)p.kprime * band_x4 / 4 + (uint64_t)p.kprime > (uint64_t)kSelCap) growth /= 2;
    const uint64_t total_tiles = (p.n_rows + BN - 1) / BN;
    uint64_t mult = (uint64_t)((double)total_tiles * 0.6180339887498949) | 1ull;
    auto gcd = [](uint64_t a, uint64_t b) { while (b) { uint64_t t = a % b; a = b; b = t; } return a; };
    while (mult > 1 && gcd(mult, total_tiles) != 1) mult += 2;
    if (total_tiles <= 2 || p.sequential_tiles) mult = 1;
    mult %= total_tiles > 0 ? total_tiles : 1;
    if (mult == 0) mult = 1;
    uint64_t begin = 0, end = 1024 / BN;
    while (begin < total_tiles) {
        if (end > total_tiles || end + end / 4 > total_tiles) end = total_tiles;
        const uint64_t n_tiles = end - begin;
        uint64_t chunk = (n_tiles * (uint64_t)n_qtiles + (uint64_t)workers * 4 - 1) / ((uint64_t)workers * 4);
        if (chunk < 1) chunk = 1;
        if (chunk > 64) chunk = 64;
        if (p.chunk_tiles > 0) chunk = (uint64_t)p.chunk_tiles;
        if (cg == 2)
            e = launch_round<2>(p.grid, s, tq, tx, ts, (uint32_t)begin, (uint32_t)end, (uint32_t)p.n_rows, (uint32_t)total_tiles,
                                (uint32_t)mult, n_qtiles, p.n_queries, (int)chunk, thr, cnt, log, overflow, arrive, cq);
        else
            e = launch_round<1>(p.grid, s, tq, tx, ts, (uint32_t)begin, (uint32_t)end, (uint32_t)p.n_rows, (uint32_t)total_tiles,
                                (uint32_t)mult, n_qtiles, p.n_queries, (int)chunk, thr, cnt, log, overflow, arrive, cq);
        if (e != cudaSuccess) return e;
#ifdef DAWN_COUNT_SLOW_PATH
        slow_path_log_kernel<<<1, 1, 0, s>>>((uint32_t)(end - begin), p.n_queries);
#endif
        const bool last = end >= total_tiles;
        select_i8_kernel<<<qp, kSelThreads, 0, s>>>(log, cnt, kept, thr, overflow, kSelCap, p.kprime, p.arena, p.queries,
                                                    p.n_queries, s1, e1, p.limit_score, p.eps_scale, p.labels,
                                                    last ? p.final_lists : nullptr, arrive, p.rescore_f16);
        launches += 2;
        begin = end;
        end = end * growth;
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (p.overflow_out) *p.overflow_out = overflow;
    if (p.launches_out) *p.launches_out = launches;
    return cudaSuccess;
}

}  // namespace dawn

#ifdef DAWN_COUNT_SLOW_PATH
// The measurement build's log on the current device: copies up to `cap` entries of 4 u64 into out, returns the number logged
// (-1 on a CUDA error); reset != 0 then empties it.
extern "C" int dawn_debug_slow_path_log(unsigned long long *out, int cap, int reset) {
    unsigned int n = 0;
    if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpyFromSymbol(&n, dawn::g_slow_log_n, sizeof n) != cudaSuccess) return -1;
    const int m = (int)n < cap ? (int)n : cap;
    if (m > 0 && cudaMemcpyFromSymbol(out, dawn::g_slow_log, (size_t)m * 4 * sizeof(unsigned long long)) != cudaSuccess) return -1;
    if (reset) {
        const unsigned int zero = 0;
        if (cudaMemcpyToSymbol(dawn::g_slow_log_n, &zero, sizeof zero) != cudaSuccess) return -1;
    }
    return (int)n;
}
#endif
