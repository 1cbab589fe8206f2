// remove.cu -- device side of dawn_index_remove_batch: rows whose label is in a requested set are compacted out of the
// corpus in place.  Exact search does not depend on row order, so instead of tombstones that every search kernel would have
// to test, the last rows of the corpus move into the holes and the size shrinks:
//
//   build  the m requested labels -> open-addressing hash table (>= 2m slots), O(m)
//   mark   one pass over labels[0, n): a bit per row (one 32-bit word per 32 rows) and a count per 8192-row tile
//   scan   one CTA: tile prefix sums, r = rows to remove, h = flagged rows below n - r
//   pair   hole i = i-th flagged row in [0, n - r), donor i = i-th unflagged row in [n - r, n), both ascending
//   move   one warp per pair: every byte the donor owns is copied into the hole
//
// Holes and donors pair in ascending row order, so the same calls always give the same placement (and a byte-identical
// save file).  The host side (dawn_index.cu) runs build..pair before taking the exclusive corpus lock -- they only read the
// label table -- and move plus the size update under it.
#include "dawn_common.cuh"

namespace dawn {

namespace {

constexpr int kTileRows = 8192;                 // rows per mark / pair CTA: 8 warps x 32 words x 32 rows
constexpr int kTileWords = kTileRows / 32;
constexpr uint64_t kEmptySlot = kNoLabel;       // the label ~0 itself is kept in a flag word instead of the table

inline size_t align256(size_t b) { return (b + 255) / 256 * 256; }

struct Layout {
    size_t table_slots, n_tiles;
    size_t off_table, off_words, off_tile_cnt, off_tile_pre, off_meta, bytes;
};

Layout layout_of(size_t m, size_t n) {
    Layout L;
    L.table_slots = 64;
    while (L.table_slots < 2 * m) L.table_slots <<= 1;
    L.n_tiles = (n + kTileRows - 1) / kTileRows;
    L.off_table = 0;
    L.off_words = align256(L.off_table + L.table_slots * sizeof(uint64_t));
    L.off_tile_cnt = align256(L.off_words + L.n_tiles * kTileWords * sizeof(uint32_t));
    L.off_tile_pre = align256(L.off_tile_cnt + L.n_tiles * sizeof(uint32_t));
    L.off_meta = align256(L.off_tile_pre + L.n_tiles * sizeof(uint32_t));
    L.bytes = align256(L.off_meta + 4 * sizeof(uint32_t));
    return L;
}

// meta words: [0] r (rows to remove), [1] h (holes = pairs), [2] 1 if the label ~0 was requested
__global__ void __launch_bounds__(256) remove_build_kernel(const uint64_t *__restrict__ req, size_t m, uint64_t *table,
                                                           uint64_t mask, uint32_t *__restrict__ meta) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
        const uint64_t key = req[i];
        if (key == kEmptySlot) {
            meta[2] = 1u;
            continue;
        }
        uint64_t slot = mix64(key) & mask;
        while (true) {  // at most half the slots are ever taken, so an empty one is always found
            const unsigned long long prev = atomicCAS(reinterpret_cast<unsigned long long *>(table + slot),
                                                      (unsigned long long)kEmptySlot, (unsigned long long)key);
            if (prev == kEmptySlot || prev == key) break;  // inserted, or a repeat of a label already in the set
            slot = (slot + 1) & mask;
        }
    }
}

__device__ __forceinline__ bool in_set(uint64_t key, const uint64_t *__restrict__ table, uint64_t mask, bool has_max) {
    if (key == kEmptySlot) return has_max;
    uint64_t slot = mix64(key) & mask;
    while (true) {
        const uint64_t v = __ldg(reinterpret_cast<const unsigned long long *>(table + slot));
        if (v == key) return true;
        if (v == kEmptySlot) return false;
        slot = (slot + 1) & mask;
    }
}

// One CTA per tile of 8192 rows; warp w owns rows [w*1024, (w+1)*1024) of the tile, one ballot word per 32 rows.
__global__ void __launch_bounds__(256) remove_mark_kernel(const uint64_t *__restrict__ labels, size_t n,
                                                          const uint64_t *__restrict__ table, uint64_t mask,
                                                          const uint32_t *__restrict__ meta, uint32_t *__restrict__ words,
                                                          uint32_t *__restrict__ tile_cnt) {
    __shared__ uint32_t s_cnt[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool has_max = meta[2] != 0;
    const size_t word0 = (size_t)blockIdx.x * kTileWords + (size_t)warp * 32;
    uint32_t cnt = 0, mine = 0;
    for (int it0 = 0; it0 < 32; it0 += 8) {
        uint64_t lab[8];  // eight loads in flight per lane before the first probe
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const size_t row = (word0 + it0 + j) * 32 + lane;
            lab[j] = row < n ? __ldg(reinterpret_cast<const unsigned long long *>(labels + row)) : 0ull;
        }
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const size_t row = (word0 + it0 + j) * 32 + lane;
            const uint32_t b = __ballot_sync(0xffffffffu, row < n && in_set(lab[j], table, mask, has_max));
            cnt += __popc(b);
            if (lane == it0 + j) mine = b;
        }
    }
    words[word0 + lane] = mine;  // one coalesced store of the warp's 32 words
    if (lane == 0) s_cnt[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) t += s_cnt[w];
        tile_cnt[blockIdx.x] = t;
    }
}

// One CTA of 1024 threads: exclusive prefix of the tile counts, r = their sum, h = flagged rows in [0, n - r).
__global__ void __launch_bounds__(1024) remove_scan_kernel(const uint32_t *__restrict__ tile_cnt, size_t n_tiles,
                                                           const uint32_t *__restrict__ words, size_t n,
                                                           uint32_t *__restrict__ tile_pre, uint32_t *__restrict__ meta) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_total;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t per = (n_tiles + 1023) / 1024;
    const size_t a = (size_t)tid * per, b = a + per < n_tiles ? a + per : n_tiles;
    uint32_t local = 0;
    for (size_t i = a; i < b; i++) local += tile_cnt[i];
    uint32_t incl = local;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = s_warp[lane], wi = w;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, wi, off);
            if (lane >= off) wi += v;
        }
        s_warp[lane] = wi - w;  // exclusive prefix of the warp sums
        if (lane == 31) s_total = wi;
    }
    __syncthreads();
    uint32_t run = s_warp[warp] + incl - local;
    for (size_t i = a; i < b; i++) {
        tile_pre[i] = run;
        run += tile_cnt[i];
    }
    __syncthreads();  // tile_pre of the cut's tile is read below
    const uint32_t r = s_total;
    const size_t cut = n - r;
    // h = tile_pre[cut's tile] + set bits of that tile's words before the cut
    const size_t t = cut / kTileRows;
    uint32_t part = 0;
    if (t < n_tiles) {
        const size_t w0 = t * kTileWords, wc = cut / 32;
        for (size_t w = w0 + tid; w <= wc && w < w0 + kTileWords; w += blockDim.x) {
            const uint32_t bits = words[w];
            const uint32_t keep = w < wc ? 0xffffffffu : (cut % 32 ? (1u << (cut % 32)) - 1u : 0u);
            part += __popc(bits & keep);
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
    __syncthreads();
    if (lane == 0) s_warp[warp] = part;
    __syncthreads();
    if (tid == 0) {
        uint32_t h = t < n_tiles ? tile_pre[t] : r;
        for (int w = 0; w < 32; w++) h += s_warp[w];
        meta[0] = r;
        meta[1] = h;
    }
}

// One CTA per tile, one lane per word.  The rank of a flagged row is the number of flagged rows before it (tile prefix +
// word prefix + bits below it in its word); a hole's pair index is that rank, a donor's is its rank among the unflagged rows
// of [cut, n): (row - cut) - (flagged rows in [cut, row)) = (row - cut) - (rank - h).
__global__ void __launch_bounds__(256) remove_pair_kernel(const uint32_t *__restrict__ words, const uint32_t *__restrict__ tile_pre,
                                                          size_t n, size_t cut, uint32_t h, uint32_t *__restrict__ holes,
                                                          uint32_t *__restrict__ donors) {
    __shared__ uint32_t s_warp[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t w = (size_t)blockIdx.x * kTileWords + threadIdx.x;
    const uint32_t bits = words[w];
    const uint32_t pc = __popc(bits);
    uint32_t incl = pc;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t pre = tile_pre[blockIdx.x] + incl - pc;
    for (int i = 0; i < warp; i++) pre += s_warp[i];
    const size_t base = w * 32;
    auto low = [](size_t k) -> uint32_t { return k >= 32 ? 0xffffffffu : (1u << k) - 1u; };  // bits [0, k)
    uint32_t hb = base >= cut ? 0u : bits & low(cut - base);  // flagged rows below the cut
    while (hb) {
        const int j = __ffs(hb) - 1;
        hb &= hb - 1;
        holes[pre + __popc(bits & ((1u << j) - 1u))] = (uint32_t)(base + j);
    }
    const uint32_t region = (base + 32 <= cut || base >= n) ? 0u : low(n - base) & ~(base >= cut ? 0u : low(cut - base));
    uint32_t db = ~bits & region;  // unflagged rows in [cut, n)
    while (db) {
        const int j = __ffs(db) - 1;
        db &= db - 1;
        const size_t row = base + j;
        const uint32_t rank = pre + __popc(bits & ((1u << j) - 1u));
        donors[(uint32_t)(row - cut) - (rank - h)] = (uint32_t)row;
    }
}

// Lanes 0-23 of a warp move row `from_row` of the blocked int8 arena `from` (24 x 16 B) to row `to_row` of `to`; lane 24
// moves its scale.
__device__ inline void move_i8_row(const uint8_t *from, size_t from_row, uint8_t *to, size_t to_row, int lane) {
    if (lane < 24) {
        const uint4 v = *reinterpret_cast<const uint4 *>(from + i8_row_offset(from_row) + lane * 16);
        *reinterpret_cast<uint4 *>(to + i8_row_offset(to_row) + lane * 16) = v;
    } else if (lane == 24) {
        *reinterpret_cast<float *>(to + i8_scale_offset(to_row)) = *reinterpret_cast<const float *>(from + i8_scale_offset(from_row));
    }
}

// One warp per (hole, donor) pair.  Holes lie below the cut and donors above it, so no pair reads what another writes.
__global__ void __launch_bounds__(256) remove_move_kernel(RemoveMove p) {
    const int lane = threadIdx.x & 31;
    const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < p.n_pairs; i += n_warps) {
        const size_t hole = p.holes[i], donor = p.donors[i];
        if (p.i8) {  // DAWN_SCALAR_I8: the int8 row and its scale in the blocked layout
            move_i8_row(p.arena, donor, p.arena, hole, lane);
        } else {  // the fp16 row: 48 x 16 B
            const uint4 *src = reinterpret_cast<const uint4 *>(p.arena + donor * kRowBytesF16);
            uint4 *dst = reinterpret_cast<uint4 *>(p.arena + hole * kRowBytesF16);
            dst[lane] = src[lane];
            if (lane < 16) dst[32 + lane] = src[32 + lane];
        }
        if (p.corpus32) {  // DAWN_SCALAR_F32: the vector as given, 96 x 16 B
            const uint4 *src = reinterpret_cast<const uint4 *>(p.corpus32 + donor * kDim);
            uint4 *dst = reinterpret_cast<uint4 *>(p.corpus32 + hole * kDim);
#pragma unroll
            for (int j = 0; j < 3; j++) dst[lane + 32 * j] = src[lane + 32 * j];
        }
        if (p.shadow)  // the int8 shadow row keeps ITS OWN scale, which its kappa bound was measured with
            move_i8_row(p.shadow, donor, p.shadow, hole, lane);
        if (lane == 31) p.labels[hole] = p.labels[donor];
    }
}

// One warp per row.  src (staged source blocks) and dst are different buffers.
__global__ void __launch_bounds__(256) reblock_i8_kernel(const uint8_t *__restrict__ src, size_t src_first, uint8_t *__restrict__ dst,
                                                         size_t dst_first, size_t n) {
    const int lane = threadIdx.x & 31;
    const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += n_warps)
        move_i8_row(src, src_first + i, dst, dst_first + i, lane);
}

inline unsigned grid_for(size_t items, size_t per_block) {
    size_t blocks = (items + per_block - 1) / per_block;
    if (blocks > 148 * 8) blocks = 148 * 8;
    return (unsigned)(blocks ? blocks : 1);
}

}  // namespace

size_t remove_scratch_bytes(size_t m, size_t n) { return layout_of(m, n).bytes; }

cudaError_t launch_remove_mark(const uint64_t *d_req, size_t m, const uint64_t *labels, size_t n, void *scratch, uint32_t *meta_out,
                               cudaStream_t s) {
    if (m == 0 || n == 0 || n > 0xFFFFFFF0ull) return cudaErrorInvalidValue;
    const Layout L = layout_of(m, n);
    uint8_t *base = static_cast<uint8_t *>(scratch);
    uint64_t *table = reinterpret_cast<uint64_t *>(base + L.off_table);
    uint32_t *words = reinterpret_cast<uint32_t *>(base + L.off_words);
    uint32_t *tile_cnt = reinterpret_cast<uint32_t *>(base + L.off_tile_cnt);
    uint32_t *tile_pre = reinterpret_cast<uint32_t *>(base + L.off_tile_pre);
    uint32_t *meta = reinterpret_cast<uint32_t *>(base + L.off_meta);
    cudaError_t e = cudaMemsetAsync(table, 0xFF, L.table_slots * sizeof(uint64_t), s);
    if (e == cudaSuccess) e = cudaMemsetAsync(meta, 0, 4 * sizeof(uint32_t), s);
    if (e != cudaSuccess) return e;
    const uint64_t mask = L.table_slots - 1;
    remove_build_kernel<<<grid_for(m, 256), 256, 0, s>>>(d_req, m, table, mask, meta);
    remove_mark_kernel<<<(unsigned)L.n_tiles, 256, 0, s>>>(labels, n, table, mask, meta, words, tile_cnt);
    remove_scan_kernel<<<1, 1024, 0, s>>>(tile_cnt, L.n_tiles, words, n, tile_pre, meta);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    return cudaMemcpyAsync(meta_out, meta, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s);
}

cudaError_t launch_remove_pair(const void *scratch, size_t m, size_t n, uint32_t r, uint32_t h, uint32_t *holes, uint32_t *donors,
                               cudaStream_t s) {
    if (h == 0) return cudaSuccess;
    const Layout L = layout_of(m, n);
    const uint8_t *base = static_cast<const uint8_t *>(scratch);
    remove_pair_kernel<<<(unsigned)L.n_tiles, kTileWords, 0, s>>>(reinterpret_cast<const uint32_t *>(base + L.off_words),
                                                                  reinterpret_cast<const uint32_t *>(base + L.off_tile_pre), n,
                                                                  n - r, h, holes, donors);
    return cudaGetLastError();
}

cudaError_t launch_remove_move(const RemoveMove &p, cudaStream_t s) {
    if (p.n_pairs == 0) return cudaSuccess;
    remove_move_kernel<<<grid_for(p.n_pairs, 8), 256, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_reblock_i8(const uint8_t *src, size_t src_first, uint8_t *dst, size_t dst_first, size_t n, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    reblock_i8_kernel<<<grid_for(n, 8), 256, 0, s>>>(src, src_first, dst, dst_first, n);
    return cudaGetLastError();
}

}  // namespace dawn
