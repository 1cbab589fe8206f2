// ingest.cu -- K1: moving page vectors into (and out of) the device-resident fp16 corpus.
//
// Replaces what usearch's Index::add does with the vector payload
// (/root/reference/src/search/search_provider.rs:149,284): the reference stores the f32
// vector inside the HNSW graph; here it is rounded once to fp16 (round to nearest even)
// and appended to the corpus arena.  The caller's normalisation gate
// (src/search/vector.rs:185-192, applied at search_provider.rs:265) stays on the host
// side of the boundary, exactly as in the reference, so the conversion is elementwise
// and bit-exact against oracle/dawn_oracle.c:dawn_oracle_store_f16.
//
// All three kernels are pure streaming: 128-bit accesses, grid-stride, HBM-bound.
#include "dawn_common.cuh"

namespace dawn {

namespace {

// saturate: the selection copy of DAWN_SCALAR_F32 rows keeps every non-NaN value at most +-65504, so that a value out of the
// fp16 range still ranks its row near where it belongs (an inf copy would give inf - inf = NaN and drop the row).
__device__ __forceinline__ float sat_f16(float v) { return v < -65504.f ? -65504.f : v > 65504.f ? 65504.f : v; }

__global__ void __launch_bounds__(256) ingest_f16_kernel(const float4 *__restrict__ src,
                                                         uint4 *__restrict__ dst, size_t n_vec8, bool saturate) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec8; i += stride) {
        float4 a = src[2 * i], b = src[2 * i + 1];
        if (saturate) {
            a = make_float4(sat_f16(a.x), sat_f16(a.y), sat_f16(a.z), sat_f16(a.w));
            b = make_float4(sat_f16(b.x), sat_f16(b.y), sat_f16(b.z), sat_f16(b.w));
        }
        __half2 h0 = __floats2half2_rn(a.x, a.y), h1 = __floats2half2_rn(a.z, a.w);
        __half2 h2 = __floats2half2_rn(b.x, b.y), h3 = __floats2half2_rn(b.z, b.w);
        uint4 o;
        o.x = *reinterpret_cast<uint32_t *>(&h0);
        o.y = *reinterpret_cast<uint32_t *>(&h1);
        o.z = *reinterpret_cast<uint32_t *>(&h2);
        o.w = *reinterpret_cast<uint32_t *>(&h3);
        dst[i] = o;
    }
}

// One warp per row.  Lane l owns columns [8l, 8l+8) and [256+4l, 256+4l+4): the same
// split the scan kernel uses, so stores are one 128-bit and one 64-bit access per lane.
__global__ void __launch_bounds__(256) synth_f16_kernel(__half *__restrict__ dst, uint64_t seed,
                                                        uint64_t first_row, size_t n_rows) {
    const int lane = threadIdx.x & 31;
    size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = warp; r < n_rows; r += n_warps) {
        uint64_t row = first_row + r;
        int32_t raw[12];
        long long sumsq = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) raw[j] = synth_raw(seed, row, lane * 8 + j);
#pragma unroll
        for (int j = 0; j < 4; j++) raw[8 + j] = synth_raw(seed, row, 256 + lane * 4 + j);
#pragma unroll
        for (int j = 0; j < 12; j++) sumsq += (long long)raw[j] * raw[j];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) sumsq += __shfl_xor_sync(0xffffffffu, sumsq, off);
        if (sumsq == 0) {  // cannot happen for a real hash; mirrors the oracle's guard
            if (lane == 0) raw[0] = 1;
            sumsq = 1;
        }
        double inv = 1.0 / sqrt((double)sumsq);
        __half h[12];
#pragma unroll
        for (int j = 0; j < 12; j++) h[j] = __float2half_rn((float)((double)raw[j] * inv));
        __half *out = dst + r * kDim;
        *reinterpret_cast<uint4 *>(out + lane * 8) = *reinterpret_cast<uint4 *>(&h[0]);
        *reinterpret_cast<uint2 *>(out + 256 + lane * 4) = *reinterpret_cast<uint2 *>(&h[8]);
    }
}

// The synthetic rows as f32 (one warp per row, same column split as synth_f16_kernel).
__global__ void __launch_bounds__(256) synth_f32_kernel(float *__restrict__ dst, uint64_t seed, uint64_t first_row,
                                                        size_t n_rows) {
    const int lane = threadIdx.x & 31;
    size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = warp; r < n_rows; r += n_warps) {
        uint64_t row = first_row + r;
        int32_t raw[12];
        long long sumsq = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) raw[j] = synth_raw(seed, row, lane * 8 + j);
#pragma unroll
        for (int j = 0; j < 4; j++) raw[8 + j] = synth_raw(seed, row, 256 + lane * 4 + j);
#pragma unroll
        for (int j = 0; j < 12; j++) sumsq += (long long)raw[j] * raw[j];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) sumsq += __shfl_xor_sync(0xffffffffu, sumsq, off);
        if (sumsq == 0) {
            if (lane == 0) raw[0] = 1;
            sumsq = 1;
        }
        double inv = 1.0 / sqrt((double)sumsq);
        float x[12];
#pragma unroll
        for (int j = 0; j < 12; j++) x[j] = (float)((double)raw[j] * inv);
        float *out = dst + r * kDim;
        *reinterpret_cast<float4 *>(out + lane * 8) = make_float4(x[0], x[1], x[2], x[3]);
        *reinterpret_cast<float4 *>(out + lane * 8 + 4) = make_float4(x[4], x[5], x[6], x[7]);
        *reinterpret_cast<float4 *>(out + 256 + lane * 4) = make_float4(x[8], x[9], x[10], x[11]);
    }
}

__global__ void __launch_bounds__(128) gather_f32_kernel(const __half *__restrict__ corpus,
                                                         const uint32_t *__restrict__ rows, size_t n,
                                                         float *__restrict__ out) {
    size_t i = blockIdx.x;
    if (i >= n) return;
    const __half *src = corpus + (size_t)rows[i] * kDim;
    for (int c = threadIdx.x; c < kDim; c += blockDim.x) out[i * kDim + c] = __half2float(src[c]);
}

// ---- int8 storage (K4): per-row scale = absmax/127 (1 if the row is all zero), q = round half away
// from zero (the reference's rounding, src/search/vector.rs:30-32), clamped to [-127,127].
// Bit-exact against oracle/dawn_oracle.c:dawn_oracle_store_i8: max is order independent and the
// divisions are IEEE.  One warp per row; lane l owns columns [8l,8l+8) and [256+4l,256+4l+4).
__device__ __forceinline__ void quantize_row_i8(const float (&x)[12], uint8_t *arena, size_t dst_row, int lane) {
    float amax = 0.f;
#pragma unroll
    for (int j = 0; j < 12; j++) amax = fmaxf(amax, fabsf(x[j]));
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, off));
    const float scale = amax > 0.f ? __fdiv_rn(amax, 127.0f) : 1.0f;
    int8_t qv[12];
#pragma unroll
    for (int j = 0; j < 12; j++) {
        float q = roundf(__fdiv_rn(x[j], scale));
        q = q == q ? fminf(127.f, fmaxf(-127.f, q)) : 0.f;  // a NaN quotient (NaN, or inf / inf) stores 0, as Rust's `as` does
        qv[j] = (int8_t)q;
    }
    uint8_t *row = arena + i8_row_offset(dst_row);
    *reinterpret_cast<uint2 *>(row + lane * 8) = *reinterpret_cast<uint2 *>(&qv[0]);
    *reinterpret_cast<uint32_t *>(row + 256 + lane * 4) = *reinterpret_cast<uint32_t *>(&qv[8]);
    if (lane == 0) *reinterpret_cast<float *>(arena + i8_scale_offset(dst_row)) = scale;
}

__global__ void __launch_bounds__(256) ingest_i8_kernel(const float *__restrict__ src, uint8_t *__restrict__ arena,
                                                        size_t first_row, size_t n_rows) {
    const int lane = threadIdx.x & 31;
    size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = warp; r < n_rows; r += n_warps) {
        const float *in = src + r * kDim;
        float x[12];
        const float4 a = *reinterpret_cast<const float4 *>(in + lane * 8);
        const float4 b = *reinterpret_cast<const float4 *>(in + lane * 8 + 4);
        const float4 c = *reinterpret_cast<const float4 *>(in + 256 + lane * 4);
        x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
        x[8] = c.x; x[9] = c.y; x[10] = c.z; x[11] = c.w;
        quantize_row_i8(x, arena, first_row + r, lane);
    }
}

__global__ void __launch_bounds__(256) synth_i8_kernel(uint8_t *__restrict__ arena, size_t dst_first_row, uint64_t seed,
                                                       uint64_t first_row, size_t n_rows) {
    const int lane = threadIdx.x & 31;
    size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = warp; r < n_rows; r += n_warps) {
        uint64_t row = first_row + r;
        int32_t raw[12];
        long long sumsq = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) raw[j] = synth_raw(seed, row, lane * 8 + j);
#pragma unroll
        for (int j = 0; j < 4; j++) raw[8 + j] = synth_raw(seed, row, 256 + lane * 4 + j);
#pragma unroll
        for (int j = 0; j < 12; j++) sumsq += (long long)raw[j] * raw[j];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) sumsq += __shfl_xor_sync(0xffffffffu, sumsq, off);
        if (sumsq == 0) {
            if (lane == 0) raw[0] = 1;
            sumsq = 1;
        }
        double inv = 1.0 / sqrt((double)sumsq);
        float x[12];
#pragma unroll
        for (int j = 0; j < 12; j++) x[j] = (float)((double)raw[j] * inv);
        quantize_row_i8(x, arena, dst_first_row + r, lane);
    }
}

__global__ void __launch_bounds__(128) gather_f32_i8_kernel(const uint8_t *__restrict__ arena,
                                                            const uint32_t *__restrict__ rows, size_t n,
                                                            float *__restrict__ out) {
    size_t i = blockIdx.x;
    if (i >= n) return;
    const size_t row = rows[i];
    const int8_t *src = reinterpret_cast<const int8_t *>(arena + i8_row_offset(row));
    const float scale = *reinterpret_cast<const float *>(arena + i8_scale_offset(row));
    for (int c = threadIdx.x; c < kDim; c += blockDim.x) out[i * kDim + c] = __fmul_rn((float)src[c], scale);
}

}  // namespace

cudaError_t launch_ingest_i8(const float *src_f32, uint8_t *arena, size_t first_row, size_t n_rows, cudaStream_t s) {
    if (n_rows == 0) return cudaSuccess;
    size_t blocks = (n_rows + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    ingest_i8_kernel<<<(unsigned)blocks, 256, 0, s>>>(src_f32, arena, first_row, n_rows);
    return cudaGetLastError();
}

cudaError_t launch_synth_i8(uint8_t *arena, size_t dst_first_row, uint64_t seed, uint64_t first_row, size_t n_rows,
                            cudaStream_t s) {
    if (n_rows == 0) return cudaSuccess;
    size_t blocks = (n_rows + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    synth_i8_kernel<<<(unsigned)blocks, 256, 0, s>>>(arena, dst_first_row, seed, first_row, n_rows);
    return cudaGetLastError();
}

cudaError_t launch_gather_f32_i8(const uint8_t *arena, const uint32_t *rows, size_t n, float *out, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    gather_f32_i8_kernel<<<(unsigned)n, 128, 0, s>>>(arena, rows, n, out);
    return cudaGetLastError();
}

cudaError_t launch_ingest_f16(const float *src_f32, __half *dst, size_t n_rows, cudaStream_t s, bool saturate) {
    if (n_rows == 0) return cudaSuccess;
    size_t n_vec8 = n_rows * (kDim / 8);
    size_t blocks = (n_vec8 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    ingest_f16_kernel<<<(unsigned)blocks, 256, 0, s>>>(reinterpret_cast<const float4 *>(src_f32),
                                                      reinterpret_cast<uint4 *>(dst), n_vec8, saturate);
    return cudaGetLastError();
}

cudaError_t launch_synth_f16(__half *dst, uint64_t seed, uint64_t first_row, size_t n_rows,
                             cudaStream_t s) {
    if (n_rows == 0) return cudaSuccess;
    size_t blocks = (n_rows + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    synth_f16_kernel<<<(unsigned)blocks, 256, 0, s>>>(dst, seed, first_row, n_rows);
    return cudaGetLastError();
}

cudaError_t launch_synth_f32(float *dst, uint64_t seed, uint64_t first_row, size_t n_rows, cudaStream_t s) {
    if (n_rows == 0) return cudaSuccess;
    size_t blocks = (n_rows + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    synth_f32_kernel<<<(unsigned)blocks, 256, 0, s>>>(dst, seed, first_row, n_rows);
    return cudaGetLastError();
}

cudaError_t launch_gather_f32(const __half *corpus, const uint32_t *rows, size_t n, float *out,
                              cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    gather_f32_kernel<<<(unsigned)n, 128, 0, s>>>(corpus, rows, n, out);
    return cudaGetLastError();
}

}  // namespace dawn
