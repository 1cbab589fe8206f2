/*
 * dawn_oracle.c -- scalar CPU restatement of the DawnSearch vector top-k hot path.
 *
 * TEST INFRASTRUCTURE ONLY (see dawn_oracle.h).  PARITY UNPINNED by the reference:
 * it has no tests or golden vectors for this path; each function below cites the
 * reference lines it follows (paths relative to /root/reference/).
 *
 * Build with -ffp-contract=off: the reference is Rust, which never fuses a*b+c,
 * so every multiply and every add below must round separately.
 */
#include "dawn_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define EM DAWN_ORACLE_EM_LEN

/* ------------------------------------------------------------------ vector.rs */

/* src/search/vector.rs:95-97 -- zip(a,b).map((a-b).powf(2.0)).sum(), f32, in index order. */
float dawn_oracle_distance_l2sq(const float *a, const float *b) {
    float acc = 0.0f;
    for (int i = 0; i < EM; i++) {
        float d = a[i] - b[i];
        acc += d * d;
    }
    return acc;
}

/* src/search/vector.rs:99-101 -- zip(a,b).map(a*b).sum(). */
float dawn_oracle_distance_ip(const float *a, const float *b) {
    float acc = 0.0f;
    for (int i = 0; i < EM; i++) acc += a[i] * b[i];
    return acc;
}

/* src/search/vector.rs:128-134 -- result += a[i]*b[i]; 1.0 - result. */
float dawn_oracle_distance_cosine(const float *a, const float *b) {
    return 1.0f - dawn_oracle_distance_ip(a, b);
}

/* src/search/vector.rs:181-183 */
float dawn_oracle_vector_length(const float *v) {
    float zero[EM];
    memset(zero, 0, sizeof zero);
    return sqrtf(dawn_oracle_distance_l2sq(v, zero));
}

/* src/search/vector.rs:185-192 -- MAX_VECTOR_DELTA = 0.01 */
int dawn_oracle_is_normalized(const float *v) {
    float l = dawn_oracle_vector_length(v);
    if (!isfinite(l)) return 0;
    return l > 1.0f - 0.01f && l < 1.0f + 0.01f;
}

/* src/search/vector.rs:194-197 */
void dawn_oracle_normalize(float *v) {
    float acc = 0.0f;
    for (int i = 0; i < EM; i++) acc += v[i] * v[i];
    float length = sqrtf(acc);
    for (int i = 0; i < EM; i++) v[i] /= length;
}

/* src/search/vector.rs:30-32 -- Rust f32::round is half-away-from-zero, `as i16` saturates
 * and maps NaN to 0. */
int16_t dawn_oracle_f32_to_i16(float x) {
    float r = roundf(x * 32767.0f);
    if (r != r) return 0;
    if (r >= 32767.0f) return 32767;
    if (r <= -32768.0f) return -32768;
    return (int16_t)r;
}

/* src/search/vector.rs:105-109 */
uint64_t dawn_oracle_distance_i16(const int16_t *a, const int16_t *b) {
    int64_t acc = 0;
    for (int i = 0; i < EM; i++) {
        int64_t d = (int64_t)a[i] - (int64_t)b[i];
        acc += d * d;
    }
    return (uint64_t)acc;
}

/* src/search/vector.rs:110-115 -- i64::MAX - sum(a*b) */
uint64_t dawn_oracle_distance_ip_i16(const int16_t *a, const int16_t *b) {
    int64_t acc = 0;
    for (int i = 0; i < EM; i++) acc += (int64_t)a[i] * (int64_t)b[i];
    return (uint64_t)(INT64_MAX - acc);
}

/* src/search/vector.rs:149-155 */
float dawn_oracle_distance_reduced(const float *a, const float *b) {
    uint32_t acc = 0;
    for (int i = 0; i < EM; i++) {
        int32_t d = (int32_t)dawn_oracle_f32_to_i16(a[i]) - (int32_t)dawn_oracle_f32_to_i16(b[i]);
        acc += (uint32_t)(d * d);
    }
    return (float)acc;
}

/* src/search/vector.rs:157-163 */
uint32_t dawn_oracle_distance_i8(const int8_t *a, const int8_t *b) {
    uint32_t acc = 0;
    for (int i = 0; i < EM; i++) {
        int32_t d = (int32_t)a[i] - (int32_t)b[i];
        acc += (uint32_t)(d * d);
    }
    return acc;
}

/* src/search/vector.rs:74-86 -- `as i32` truncates toward zero (saturating). */
void dawn_oracle_to24(const float *v, uint8_t *out) {
    for (int i = 0; i < EM; i++) {
        double t = (((double)v[i] + 1.0) / 2.0) * (double)0x7FFFFF;
        int32_t x;
        if (t != t) x = 0;
        else if (t >= 2147483647.0) x = INT32_MAX;
        else if (t <= -2147483648.0) x = INT32_MIN;
        else x = (int32_t)t;
        out[i * 3 + 0] = (uint8_t)(x & 0xFF);
        out[i * 3 + 1] = (uint8_t)((x >> 8) & 0xFF);
        out[i * 3 + 2] = (uint8_t)((x >> 16) & 0xFF);
    }
}

/* src/search/vector.rs:52-72.  The "sign extend" branch ORs 0xFF into the LOW byte
 * (`v |= 0xFF`); that is what the reference does, so it is restated as is.  It cannot
 * fire on to24's own output (values lie in [0, 0x7FFFFF]). */
int dawn_oracle_from24(const uint8_t *data, float *out) {
    for (int i = 0; i < EM; i++) {
        int32_t v = 0;
        v |= (int32_t)data[i * 3];
        v |= (int32_t)data[i * 3 + 1] << 8;
        v |= (int32_t)data[i * 3 + 2] << 16;
        if ((data[i * 3 + 2] & 0x80) > 0) v |= 0xFF;
        out[i] = (float)((double)v / (double)0x7FFFFF * 2.0 - 1.0);
    }
    return dawn_oracle_is_normalized(out);
}

/* -------------------------------------------------------- stored-vector formats */

static inline uint32_t f32_bits(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    return u;
}
static inline float bits_f32(uint32_t u) {
    float x;
    memcpy(&x, &u, 4);
    return x;
}

uint16_t dawn_oracle_f32_to_f16(float x) {
    uint32_t u = f32_bits(x);
    uint32_t sign = (u >> 16) & 0x8000u;
    uint32_t absu = u & 0x7FFFFFFFu;
    if (absu >= 0x7F800000u) { /* inf / nan */
        if (absu > 0x7F800000u) return (uint16_t)(sign | 0x7E00u | ((absu >> 13) & 0x3FFu));
        return (uint16_t)(sign | 0x7C00u);
    }
    if (absu >= 0x477FF000u) return (uint16_t)(sign | 0x7C00u); /* rounds to >= 65520 -> inf */
    if (absu < 0x33000001u) return (uint16_t)sign;               /* <= 2^-25 -> +-0 (ties to even) */
    int32_t exp = (int32_t)(absu >> 23) - 127;
    uint32_t man = (absu & 0x7FFFFFu) | 0x800000u; /* 24-bit significand */
    uint32_t shift, half_exp;
    if (exp < -14) { /* subnormal half */
        shift = (uint32_t)(13 + (-14 - exp));
        half_exp = 0;
    } else {
        shift = 13;
        half_exp = (uint32_t)(exp + 15);
    }
    uint32_t q = man >> shift;
    uint32_t rem = man & ((1u << shift) - 1u);
    uint32_t halfway = 1u << (shift - 1);
    if (rem > halfway || (rem == halfway && (q & 1u))) q++;
    uint32_t h;
    if (half_exp == 0) h = q; /* may carry into exponent 1: correct */
    else h = ((half_exp - 1) << 10) + q; /* q carries the implicit bit (0x400) */
    return (uint16_t)(sign | h);
}

float dawn_oracle_f16_to_f32(uint16_t h) {
    uint32_t sign = ((uint32_t)h & 0x8000u) << 16;
    uint32_t exp = (h >> 10) & 0x1Fu;
    uint32_t man = h & 0x3FFu;
    if (exp == 0x1F) return bits_f32(sign | 0x7F800000u | (man << 13));
    if (exp == 0) {
        if (man == 0) return bits_f32(sign);
        float f = (float)man * 5.9604644775390625e-08f; /* man * 2^-24, exact */
        return sign ? -f : f;
    }
    return bits_f32(sign | ((exp + 112u) << 23) | (man << 13));
}

void dawn_oracle_store_f16(const float *rows, size_t n, uint16_t *out) {
    for (size_t i = 0; i < n * EM; i++) out[i] = dawn_oracle_f32_to_f16(rows[i]);
}

void dawn_oracle_store_i8(const float *rows, size_t n, int8_t *out, float *scales) {
    for (size_t r = 0; r < n; r++) {
        const float *x = rows + r * EM;
        float amax = 0.0f;
        for (int i = 0; i < EM; i++) {
            float a = fabsf(x[i]);
            if (a > amax) amax = a;
        }
        float scale = amax > 0.0f ? amax / 127.0f : 1.0f;
        scales[r] = scale;
        for (int i = 0; i < EM; i++) {
            float q = roundf(x[i] / scale);
            if (q != q) q = 0.0f; /* a NaN quotient (NaN or inf / inf) stores 0, as Rust's `as` does */
            if (q > 127.0f) q = 127.0f;
            if (q < -127.0f) q = -127.0f;
            out[r * EM + i] = (int8_t)q;
        }
    }
}

/* ------------------------------------------------------------ synthetic corpus */

static inline uint64_t mix64(uint64_t z) { /* splitmix64 finaliser */
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

/* Irwin-Hall(4) of 16-bit uniforms, centred: an integer in [-131070, 131070]. */
static inline int32_t synth_raw(uint64_t seed, uint64_t row, uint32_t col) {
    uint64_t h = mix64(seed + 0x9E3779B97F4A7C15ull * (row * (uint64_t)EM + col + 1));
    uint32_t s = (uint32_t)(h & 0xFFFF) + (uint32_t)((h >> 16) & 0xFFFF) +
                 (uint32_t)((h >> 32) & 0xFFFF) + (uint32_t)(h >> 48);
    return (int32_t)s - 131070;
}

void dawn_oracle_synth_row_f32(uint64_t seed, uint64_t row, float *out) {
    int32_t raw[EM];
    int64_t sumsq = 0;
    for (uint32_t c = 0; c < EM; c++) {
        raw[c] = synth_raw(seed, row, c);
        sumsq += (int64_t)raw[c] * raw[c];
    }
    if (sumsq == 0) {
        raw[0] = 1;
        sumsq = 1;
    }
    double inv = 1.0 / sqrt((double)sumsq);
    for (uint32_t c = 0; c < EM; c++) out[c] = (float)((double)raw[c] * inv);
}

void dawn_oracle_synth_rows_f16(uint64_t seed, uint64_t first_row, size_t n, uint16_t *out) {
    float tmp[EM];
    for (size_t r = 0; r < n; r++) {
        dawn_oracle_synth_row_f32(seed, first_row + r, tmp);
        for (int c = 0; c < EM; c++) out[r * EM + c] = dawn_oracle_f32_to_f16(tmp[c]);
    }
}

/* ------------------------------------------------------------------- top-k */

typedef struct {
    float score;
    uint64_t label;
    uint64_t row;
} cand_t;

/* Total order of results: distance asc, label asc, row asc, where distance is the f32
 * value 1.0f - score that is returned (vector.rs:133).  Ordering on the emitted distance
 * (rather than the score) keeps the output self-consistent and lets result lists from
 * several shards be merged from (label, distance) pairs alone, as the reference's
 * search_remote does with BestResults (src/search/search_service.rs:247-268). */
static inline int cand_better(const cand_t *a, const cand_t *b) {
    const float da = 1.0f - a->score, db = 1.0f - b->score;
    if (da != db) return da < db;
    if (a->label != b->label) return a->label < b->label;
    return a->row < b->row;
}

typedef struct {
    cand_t *v;
    size_t k, len;
} topk_t;

/* A row whose exact score is NaN is not a result: NaN has no place in the total order, and keeping it
 * would make the output depend on row order.  +-inf scores are ordered (distance -inf is best). */
static void topk_push(topk_t *t, cand_t c) {
    if (t->k == 0 || c.score != c.score) return;
    if (t->len == t->k) {
        if (!cand_better(&c, &t->v[t->len - 1])) return;
        t->len--;
    }
    size_t i = t->len;
    while (i > 0 && cand_better(&c, &t->v[i - 1])) {
        t->v[i] = t->v[i - 1];
        i--;
    }
    t->v[i] = c;
    t->len++;
}

static size_t topk_emit(topk_t *t, uint64_t *labels_out, float *distances_out) {
    for (size_t i = 0; i < t->len; i++) {
        labels_out[i] = t->v[i].label;
        distances_out[i] = 1.0f - t->v[i].score; /* vector.rs:133 */
    }
    return t->len;
}

float dawn_oracle_score_f16(const uint16_t *row, const float *query) {
    float acc = 0.0f;
    for (int i = 0; i < EM; i++) acc += query[i] * dawn_oracle_f16_to_f32(row[i]);
    return acc;
}

/* The sequential sum is a 384-long dependency chain; ROWS_IL rows are interleaved so the
 * chains overlap.  Each row's own order of operations is unchanged. */
#define ROWS_IL 8

size_t dawn_oracle_search_f16(const uint16_t *corpus, const uint64_t *labels, size_t n,
                              const float *query, size_t k, uint64_t *labels_out,
                              float *distances_out) {
    topk_t t = {(cand_t *)malloc(sizeof(cand_t) * (k ? k : 1)), k, 0};
    size_t r = 0;
    for (; r + ROWS_IL <= n; r += ROWS_IL) {
        float acc[ROWS_IL];
        for (int j = 0; j < ROWS_IL; j++) acc[j] = 0.0f;
        for (int i = 0; i < EM; i++) {
            float q = query[i];
            for (int j = 0; j < ROWS_IL; j++)
                acc[j] += q * dawn_oracle_f16_to_f32(corpus[(r + j) * EM + i]);
        }
        for (int j = 0; j < ROWS_IL; j++) {
            cand_t c = {acc[j], labels ? labels[r + j] : (uint64_t)(r + j + 1), r + j};
            topk_push(&t, c);
        }
    }
    for (; r < n; r++) {
        cand_t c = {dawn_oracle_score_f16(corpus + r * EM, query),
                    labels ? labels[r] : (uint64_t)(r + 1), r};
        topk_push(&t, c);
    }
    size_t cnt = topk_emit(&t, labels_out, distances_out);
    free(t.v);
    return cnt;
}

size_t dawn_oracle_search_f32(const float *corpus, const uint64_t *labels, size_t n,
                              const float *query, size_t k, uint64_t *labels_out,
                              float *distances_out) {
    topk_t t = {(cand_t *)malloc(sizeof(cand_t) * (k ? k : 1)), k, 0};
    for (size_t r = 0; r < n; r++) {
        cand_t c = {dawn_oracle_distance_ip(query, corpus + r * EM),
                    labels ? labels[r] : (uint64_t)(r + 1), r};
        topk_push(&t, c);
    }
    size_t cnt = topk_emit(&t, labels_out, distances_out);
    free(t.v);
    return cnt;
}

size_t dawn_oracle_search_i8(const int8_t *corpus, const float *scales, const uint64_t *labels,
                             size_t n, const float *query, size_t k, uint64_t *labels_out,
                             float *distances_out) {
    topk_t t = {(cand_t *)malloc(sizeof(cand_t) * (k ? k : 1)), k, 0};
    for (size_t r = 0; r < n; r++) {
        float acc = 0.0f;
        for (int i = 0; i < EM; i++) acc += query[i] * (float)corpus[r * EM + i];
        cand_t c = {scales[r] * acc, labels ? labels[r] : (uint64_t)(r + 1), r};
        topk_push(&t, c);
    }
    size_t cnt = topk_emit(&t, labels_out, distances_out);
    free(t.v);
    return cnt;
}

/* ------------------------------------------------------------ best_results.rs */

struct dawn_oracle_best_results {
    uint64_t *ids;
    float *dist;
    size_t len, size, worst_index;
    float worst_distance;
};

/* src/search/best_results.rs:35-43 */
dawn_oracle_best_results *dawn_oracle_best_new(size_t size) {
    dawn_oracle_best_results *b = (dawn_oracle_best_results *)calloc(1, sizeof *b);
    b->ids = (uint64_t *)malloc(sizeof(uint64_t) * (size ? size : 1));
    b->dist = (float *)malloc(sizeof(float) * (size ? size : 1));
    b->size = size;
    b->worst_distance = 0.0f; /* T::zero() */
    return b;
}

void dawn_oracle_best_free(dawn_oracle_best_results *b) {
    if (!b) return;
    free(b->ids);
    free(b->dist);
    free(b);
}

/* src/search/best_results.rs:67-69 */
static int best_contains(const dawn_oracle_best_results *b, uint64_t id) {
    for (size_t i = 0; i < b->len; i++)
        if (b->ids[i] == id) return 1;
    return 0;
}

/* src/search/best_results.rs:97-107 */
static void best_update_worst(dawn_oracle_best_results *b) {
    b->worst_index = 0;
    b->worst_distance = b->dist[0];
    for (size_t i = 1; i < b->len; i++) {
        if (b->dist[i] > b->worst_distance) {
            b->worst_distance = b->dist[i];
            b->worst_index = i;
        }
    }
}

/* src/search/best_results.rs:44-65 */
int dawn_oracle_best_insert(dawn_oracle_best_results *b, uint64_t id, float distance) {
    if (b->len < b->size) {
        if (best_contains(b, id)) return 0;
        b->ids[b->len] = id;
        b->dist[b->len] = distance;
        b->len++;
        if (b->len == b->size) best_update_worst(b);
        return 1;
    }
    if (distance < b->worst_distance) {
        if (best_contains(b, id)) return 0;
        b->ids[b->worst_index] = id;
        b->dist[b->worst_index] = distance;
        best_update_worst(b);
        return 1;
    }
    return 0;
}

/* src/search/best_results.rs:71-79 -- Vec::sort_by is a stable sort. */
void dawn_oracle_best_sort(dawn_oracle_best_results *b) {
    if (b->len == 0) return;
    for (size_t i = 1; i < b->len; i++) {
        uint64_t id = b->ids[i];
        float d = b->dist[i];
        size_t j = i;
        while (j > 0 && b->dist[j - 1] > d) {
            b->ids[j] = b->ids[j - 1];
            b->dist[j] = b->dist[j - 1];
            j--;
        }
        b->ids[j] = id;
        b->dist[j] = d;
    }
    b->worst_index = b->len - 1;
    b->worst_distance = b->dist[b->len - 1];
}

size_t dawn_oracle_best_len(const dawn_oracle_best_results *b) { return b->len; }
float dawn_oracle_best_worst_distance(const dawn_oracle_best_results *b) {
    return b->worst_distance;
}
void dawn_oracle_best_get(const dawn_oracle_best_results *b, size_t i, uint64_t *id,
                          float *distance) {
    *id = b->ids[i];
    *distance = b->dist[i];
}
