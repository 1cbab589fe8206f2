/*
 * cpu_scan.c -- threaded SIMD exact scan on host cores: the timed CPU baseline
 * ("port" kind) and the checker used where the scalar oracle would take too long.
 *
 * TEST INFRASTRUCTURE ONLY (see dawn_oracle.h); PARITY UNPINNED by the reference.
 *
 * The reference's own precedent for an exact linear scan is
 * examples_old/search.rs:45-71 (walk every stored vector, keep the best 10).  Here the
 * walk is split over threads and vectorised; because SIMD changes the order of the f32
 * additions, the SIMD pass only *selects* k+slack candidates per thread.  Candidates are
 * then re-scored with dawn_oracle_score_f16 (src/search/vector.rs:128-134 order) and
 * ranked by the oracle's total order (distance asc, label asc, row asc), so the output is
 * bit-identical to dawn_oracle_search_f16.  If the slack cannot prove that (near-ties
 * deeper than the slack), the query is re-run through the scalar oracle.
 */
#include "dawn_oracle.h"

#include <immintrin.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#define EM DAWN_ORACLE_EM_LEN
/* |simd score - sequential score| bound used by the exactness check: both are f32
 * sums of 384 products with sum |q_i x_i| <= ~1; worst case 384 * 2^-24 ~= 2.3e-5. */
#define SCAN_EPS 4.0e-5f
#define ROW_BLOCK 128

typedef struct {
    float score;
    uint64_t label;
    uint64_t row;
} cand_t;

/* candidate pass: by SIMD score (selection only) */
static inline int cand_better(const cand_t *a, const cand_t *b) {
    if (a->score != b->score) return a->score > b->score;
    if (a->label != b->label) return a->label < b->label;
    return a->row < b->row;
}

/* final ranking: the oracle's total order on the emitted distance (dawn_oracle.c) */
static inline int final_better(const cand_t *a, const cand_t *b) {
    const float da = 1.0f - a->score, db = 1.0f - b->score;
    if (da != db) return da < db;
    if (a->label != b->label) return a->label < b->label;
    return a->row < b->row;
}

typedef struct {
    cand_t *v;
    size_t k, len;
    int final;
} topk_t;

static void topk_push(topk_t *t, cand_t c) {
    if (c.score != c.score) return; /* a NaN score is not a result (dawn_oracle.c) */
    int (*better)(const cand_t *, const cand_t *) = t->final ? final_better : cand_better;
    if (t->len == t->k) {
        if (!better(&c, &t->v[t->len - 1])) return;
        t->len--;
    }
    size_t i = t->len;
    while (i > 0 && better(&c, &t->v[i - 1])) {
        t->v[i] = t->v[i - 1];
        i--;
    }
    t->v[i] = c;
    t->len++;
}

typedef void (*block_fn)(const uint16_t *rows, size_t nrows, const float *q, float *scores);

static void block_scalar(const uint16_t *rows, size_t nrows, const float *q, float *scores) {
    for (size_t r = 0; r < nrows; r++) {
        float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int i = 0; i < EM; i += 8)
            for (int j = 0; j < 8; j++) acc[j] += q[i + j] * dawn_oracle_f16_to_f32(rows[r * EM + i + j]);
        scores[r] = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
    }
}

__attribute__((target("avx2,fma,f16c"))) static void block_avx2(const uint16_t *rows, size_t nrows,
                                                                 const float *q, float *scores) {
    for (size_t r = 0; r < nrows; r++) {
        const uint16_t *x = rows + r * EM;
        __m256 a0 = _mm256_setzero_ps(), a1 = a0, a2 = a0, a3 = a0;
        for (int i = 0; i < EM; i += 32) {
            a0 = _mm256_fmadd_ps(_mm256_cvtph_ps(_mm_loadu_si128((const __m128i *)(x + i))),
                                 _mm256_loadu_ps(q + i), a0);
            a1 = _mm256_fmadd_ps(_mm256_cvtph_ps(_mm_loadu_si128((const __m128i *)(x + i + 8))),
                                 _mm256_loadu_ps(q + i + 8), a1);
            a2 = _mm256_fmadd_ps(_mm256_cvtph_ps(_mm_loadu_si128((const __m128i *)(x + i + 16))),
                                 _mm256_loadu_ps(q + i + 16), a2);
            a3 = _mm256_fmadd_ps(_mm256_cvtph_ps(_mm_loadu_si128((const __m128i *)(x + i + 24))),
                                 _mm256_loadu_ps(q + i + 24), a3);
        }
        __m256 s = _mm256_add_ps(_mm256_add_ps(a0, a1), _mm256_add_ps(a2, a3));
        __m128 lo = _mm_add_ps(_mm256_castps256_ps128(s), _mm256_extractf128_ps(s, 1));
        lo = _mm_add_ps(lo, _mm_movehl_ps(lo, lo));
        lo = _mm_add_ss(lo, _mm_shuffle_ps(lo, lo, 1));
        scores[r] = _mm_cvtss_f32(lo);
    }
}

__attribute__((target("avx512f,avx512bw,avx512vl,avx512dq,fma,f16c"))) static void block_avx512(
    const uint16_t *rows, size_t nrows, const float *q, float *scores) {
    __m512 qv[EM / 16];
    for (int i = 0; i < EM / 16; i++) qv[i] = _mm512_loadu_ps(q + 16 * i);
    for (size_t r = 0; r < nrows; r++) {
        const uint16_t *x = rows + r * EM;
        __m512 a0 = _mm512_setzero_ps(), a1 = a0, a2 = a0, a3 = a0;
        for (int i = 0; i < EM / 16; i += 4) {
            a0 = _mm512_fmadd_ps(_mm512_cvtph_ps(_mm256_loadu_si256((const __m256i *)(x + 16 * i))), qv[i], a0);
            a1 = _mm512_fmadd_ps(_mm512_cvtph_ps(_mm256_loadu_si256((const __m256i *)(x + 16 * i + 16))), qv[i + 1], a1);
            a2 = _mm512_fmadd_ps(_mm512_cvtph_ps(_mm256_loadu_si256((const __m256i *)(x + 16 * i + 32))), qv[i + 2], a2);
            a3 = _mm512_fmadd_ps(_mm512_cvtph_ps(_mm256_loadu_si256((const __m256i *)(x + 16 * i + 48))), qv[i + 3], a3);
        }
        scores[r] = _mm512_reduce_add_ps(_mm512_add_ps(_mm512_add_ps(a0, a1), _mm512_add_ps(a2, a3)));
    }
}

static block_fn pick_block_fn(void) {
    __builtin_cpu_init();
    if (__builtin_cpu_supports("avx512f") && __builtin_cpu_supports("avx512bw") &&
        __builtin_cpu_supports("avx512vl") && __builtin_cpu_supports("avx512dq"))
        return block_avx512;
    if (__builtin_cpu_supports("avx2") && __builtin_cpu_supports("fma") &&
        __builtin_cpu_supports("f16c"))
        return block_avx2;
    return block_scalar;
}

typedef struct {
    const uint16_t *corpus;
    const uint64_t *labels;
    size_t row_begin, row_end;
    const float *queries;
    size_t nq, kprime;
    topk_t *lists; /* nq lists owned by this thread */
    block_fn fn;
} job_t;

static void *scan_worker(void *arg) {
    job_t *j = (job_t *)arg;
    float scores[ROW_BLOCK];
    for (size_t r0 = j->row_begin; r0 < j->row_end; r0 += ROW_BLOCK) {
        size_t nr = j->row_end - r0 < ROW_BLOCK ? j->row_end - r0 : ROW_BLOCK;
        for (size_t qi = 0; qi < j->nq; qi++) {
            topk_t *t = &j->lists[qi];
            j->fn(j->corpus + r0 * EM, nr, j->queries + qi * EM, scores);
            float thr = t->len == t->k ? t->v[t->len - 1].score : -__builtin_inff();
            for (size_t i = 0; i < nr; i++) {
                if (scores[i] >= thr) {
                    size_t row = r0 + i;
                    cand_t c = {scores[i], j->labels ? j->labels[row] : (uint64_t)(row + 1), row};
                    topk_push(t, c);
                    if (t->len == t->k) thr = t->v[t->len - 1].score;
                }
            }
        }
    }
    return NULL;
}

int dawn_cpu_scan_threads_default(void) {
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n > 0 ? (int)n : 1;
}

int dawn_cpu_scan_f16(const uint16_t *corpus, const uint64_t *labels, size_t n,
                      const float *queries, size_t nq, size_t k, int threads,
                      uint64_t *labels_out, float *distances_out, size_t *counts_out,
                      int *certified) {
    if (certified) *certified = 1;
    if (threads <= 0) threads = dawn_cpu_scan_threads_default();
    if ((size_t)threads > n / ROW_BLOCK + 1) threads = (int)(n / ROW_BLOCK + 1);
    if (k == 0 || n == 0 || nq == 0) {
        for (size_t qi = 0; qi < nq; qi++) counts_out[qi] = 0;
        return 0;
    }
    size_t slack = k / 4 < 8 ? 8 : k / 4;
    size_t kprime = k + slack;
    block_fn fn = pick_block_fn();

    job_t *jobs = (job_t *)calloc((size_t)threads, sizeof(job_t));
    pthread_t *tids = (pthread_t *)calloc((size_t)threads, sizeof(pthread_t));
    size_t per = (n + (size_t)threads - 1) / (size_t)threads;
    per = (per + ROW_BLOCK - 1) / ROW_BLOCK * ROW_BLOCK;
    for (int t = 0; t < threads; t++) {
        job_t *j = &jobs[t];
        j->corpus = corpus;
        j->labels = labels;
        j->row_begin = (size_t)t * per < n ? (size_t)t * per : n;
        j->row_end = j->row_begin + per < n ? j->row_begin + per : n;
        j->queries = queries;
        j->nq = nq;
        j->kprime = kprime;
        j->fn = fn;
        j->lists = (topk_t *)calloc(nq, sizeof(topk_t));
        for (size_t qi = 0; qi < nq; qi++) {
            j->lists[qi].v = (cand_t *)malloc(sizeof(cand_t) * kprime);
            j->lists[qi].k = kprime;
        }
    }
    for (int t = 1; t < threads; t++) pthread_create(&tids[t], NULL, scan_worker, &jobs[t]);
    scan_worker(&jobs[0]);
    for (int t = 1; t < threads; t++) pthread_join(tids[t], NULL);

    cand_t *fin = (cand_t *)malloc(sizeof(cand_t) * (k + 1));
    for (size_t qi = 0; qi < nq; qi++) {
        const float *q = queries + qi * EM;
        topk_t out = {fin, k, 0, 1};
        for (int t = 0; t < threads; t++) {
            topk_t *l = &jobs[t].lists[qi];
            for (size_t i = 0; i < l->len; i++) {
                cand_t c = l->v[i];
                c.score = dawn_oracle_score_f16(corpus + c.row * EM, q);
                topk_push(&out, c);
            }
        }
        /* exactness check: a row a thread dropped has simd score <= that thread's weakest
         * kept candidate; it can only matter if that is within SCAN_EPS of the k-th score. */
        int ok = 1;
        if (out.len == k) {
            float dk = 1.0f - out.v[k - 1].score; /* k-th distance */
            for (int t = 0; t < threads; t++) {
                topk_t *l = &jobs[t].lists[qi];
                if (l->len == l->k && !(1.0f - (l->v[l->len - 1].score + SCAN_EPS) > dk)) ok = 0;
            }
        }
        if (!ok) {
            if (certified) *certified = 0;
            counts_out[qi] = dawn_oracle_search_f16(corpus, labels, n, q, k, labels_out + qi * k,
                                                    distances_out + qi * k);
            continue;
        }
        for (size_t i = 0; i < out.len; i++) {
            labels_out[qi * k + i] = out.v[i].label;
            distances_out[qi * k + i] = 1.0f - out.v[i].score;
        }
        counts_out[qi] = out.len;
    }
    free(fin);
    for (int t = 0; t < threads; t++) {
        for (size_t qi = 0; qi < nq; qi++) free(jobs[t].lists[qi].v);
        free(jobs[t].lists);
    }
    free(jobs);
    free(tids);
    return 0;
}
