// persist.cuh -- the pieces of save / load that dawn_index_save / _load and dawn_multi_save / _load share (dawn_index.cu).
// Internal to libdawn_b200: nothing here is exported in include/dawn_index.h.
//
// A "section" is one shard's contents in a file: uint64 labels[rows], then the stored rows exactly as the device arena
// holds them (fp16: rows x 768 B; int8: ceil(rows/8) blocks of 3104 B, unused rows and scales of a partial last block zero;
// f32: rows x 1536 B, the vectors as given).  A single-index file is a 32-byte header and one section; a multi file is a
// 4096-byte header and one page-aligned section per shard.
#pragma once

#include <stddef.h>
#include <stdint.h>

struct dawn_index;

namespace dawn {

// pwrite / pread of the whole range (false on an error or end of file).
bool pwrite_all(int fd, const void *buf, size_t n, uint64_t off);
bool pread_all(int fd, void *buf, size_t n, uint64_t off);
// Close the temporary file fd (written at tmp) and rename it to path when rc == DAWN_OK; otherwise, or when close fails,
// remove it, leaving any existing path alone.  Returns rc, or DAWN_ERR_IO (dawn_last_error says why).
int finish_file(int fd, const char *tmp, const char *path, int rc);

// Bytes of the stored rows of a section of `rows` rows (what follows its labels).
uint64_t section_payload_bytes(uint32_t scalar, uint64_t rows);

// Flush staged adds and zero the unused rows and scales of a partial last int8 block, so that the section written next is
// deterministic; *rows_out = the rows it will hold.  Takes idx->mu unless the caller already holds it.
int section_prepare(dawn_index *idx, bool caller_holds_mu, uint64_t *rows_out);

// Write rows [0, rows) of idx as a section at byte `off` of fd (pwrite), through idx's two pinned staging buffers: the D2H
// of slice i+1 overlaps the write of slice i.  Holds idx's arena pointers (corpus_mu, shared) and nothing else, so searches
// go on; the caller keeps every writer (add, remove, reserve, load, option changes) off idx until it returns.
int section_write(dawn_index *idx, int fd, uint64_t off, uint64_t rows);

struct SectionRef {
    uint64_t off;   // file offset of the labels
    uint64_t rows;
};

// A filled arena that has not been published yet (phase 1 of a load).
struct Fill {
    void *corpus = nullptr;      // fp16 rows or the blocked int8 arena
    uint64_t *labels = nullptr;
    float *corpus32 = nullptr;   // DAWN_SCALAR_F32 only
    size_t rows_alloc = 0;       // physical rows of the arena
    uint64_t rows = 0;           // rows filled
    bool in_place = false;       // the index's own (empty) arena was filled
};

// Phase 1: rows [first, first + n) of the concatenation of `secs` (in file order) into idx, read with pread.  In place when
// may_fill_in_place, idx is empty and its physical arena holds n rows; otherwise into a fresh arena.  Stored rows are
// copied, never re-quantised: int8 rows that do not start on a block boundary on both sides are staged on the device and
// re-blocked one warp per row; f32 rebuilds its fp16 selection copy.  Nothing a search reads changes.  The caller keeps
// every writer off idx.  On failure nothing needs undoing except fill_discard.
int fill_rows(dawn_index *idx, int fd, const char *path, const SectionRef *secs, size_t n_secs, uint64_t first, uint64_t n,
              bool may_fill_in_place, Fill *f);
// After a failure of this or another shard: frees a fresh arena (an in-place fill left the index empty, as it was).
void fill_discard(dawn_index *idx, Fill *f);
// Phase 2: publish the filled arena under the exclusive corpus lock: pointers, size, capacity, int8 shadow dropped, norm
// statistics reset (as after any load).  The caller holds idx->mu, or otherwise keeps every other call off idx.
void fill_commit(dawn_index *idx, Fill *f);

}  // namespace dawn
