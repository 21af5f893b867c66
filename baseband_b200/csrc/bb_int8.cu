// int8 transposed decode/encode kernels and C entry points (sm_100a).
#include <stdlib.h>
#include "bb_runtime.cuh"
#include "bb_int8.cuh"

namespace bb {

template <typename OT>
__global__ void __launch_bounds__(kI8Threads) k_int8_decode_t(const I8Geom p) {
    __shared__ __align__(16) uint8_t tile[kI8SmemBytes];
    i8_dec_load(p, tile, blockIdx.x, threadIdx.x);
    __syncthreads();
    i8_dec_store<OT>(p, tile, blockIdx.x, threadIdx.x);
}

template <typename OT>
__global__ void __launch_bounds__(kF8Threads) k_int8_decode_t64(const I8Geom p) {
    __shared__ __align__(16) uint32_t tile[kF8SmemWords];
    // knock-outs (BB_TUNE_KNOCK_I8, tools/sweep_guppi.py): which half of the
    // kernel costs what
    if (!(p.knock & 1u)) f8_dec_load(p, tile, blockIdx.x, threadIdx.x);
    __syncthreads();
    if (!(p.knock & 2u)) f8_dec_store<OT>(p, tile, blockIdx.x, threadIdx.x);
}

// Min-blocks hint of 4: lets ptxas keep eight float4 loads in flight (64
// registers) instead of serialising them to stay within 32.
template <typename S>
__global__ void __launch_bounds__(kF8Threads, 4) k_int8_encode_t64(const I8Geom p) {
    __shared__ __align__(16) uint32_t tile[kF8SmemWords];
    f8_enc_load<S>(p, tile, blockIdx.x, threadIdx.x);
    __syncthreads();
    f8_enc_store(p, tile, blockIdx.x, threadIdx.x);
}

template <typename S>
__global__ void __launch_bounds__(kI8Threads) k_int8_encode_t(const I8Geom p) {
    __shared__ __align__(16) uint8_t tile[kI8SmemBytes];
    i8_enc_load<S>(p, tile, blockIdx.x, threadIdx.x);
    __syncthreads();
    i8_enc_store(p, tile, blockIdx.x, threadIdx.x);
}

constexpr int kTFThreads = 256, kTFUnroll = 4;

template <typename OT>
__global__ void __launch_bounds__(kTFThreads) k_int8_decode_timefirst(
    const TFGeom p) {
    const uint32_t item0 = blockIdx.x * (kTFThreads * kTFUnroll) + threadIdx.x;
#pragma unroll
    for (int u = 0; u < kTFUnroll; ++u)
        tf_decode<OT>(p, blockIdx.y, item0 + u * kTFThreads);
}

template <typename S>
__global__ void __launch_bounds__(kTFThreads) k_int8_encode_timefirst(
    const TFGeom p) {
    const uint32_t item0 = blockIdx.x * (kTFThreads * kTFUnroll) + threadIdx.x;
#pragma unroll
    for (int u = 0; u < kTFUnroll; ++u)
        tf_encode<S>(p, blockIdx.y, item0 + u * kTFThreads);
}

static int fill_geom(I8Geom &g, int64_t nunit, int64_t nrow, int64_t ncol,
                     int item_nbytes, uint64_t &nblocks, bool fast = false) {
    if (item_nbytes != 1 && item_nbytes != 2)
        return set_error(BB_ERR_ARGUMENT, "item_nbytes must be 1 or 2");
    if (nunit < 0 || nrow < 1 || ncol < 1 || nrow > 0x7fffffff
        || ncol > 0x7fffffff || nunit > 0x7fffffff)
        return set_error(BB_ERR_ARGUMENT, "bad nunit/nrow/ncol");
    g.nunit = (uint32_t)nunit;
    g.nrow = (uint32_t)nrow;
    g.ncol = (uint32_t)ncol;
    g.ib = item_nbytes;
    const int rows = fast ? kF8Rows : kI8Rows;
    g.tiles_r = (uint32_t)((nrow + rows - 1) / rows);
    uint32_t tc = (fast ? kF8Words * 4 : kI8RowBytes) / item_nbytes;
    g.tiles_c = (uint32_t)((ncol + tc - 1) / tc);
    g.group = 16;
    if (const char *e = getenv("BB_I8_GROUP")) g.group = (uint32_t)atoi(e);
    g.knock = 0;
    if (const char *e = getenv("BB_TUNE_KNOCK_I8")) g.knock = (uint32_t)atoi(e);
    if (g.group < 1) g.group = 1;
    if (g.group > g.tiles_c) g.group = g.tiles_c;
    nblocks = (uint64_t)nunit * g.tiles_r * g.tiles_c;
    if (nblocks > 0x7fffffffull)
        return set_error(BB_ERR_ARGUMENT, "too many tiles for one call");
    return BB_OK;
}

template <typename OT>
static void launch_int8_decode_t(const I8Geom &g, uint64_t nblocks, bool fast,
                                 cudaStream_t s) {
    if (fast)
        k_int8_decode_t64<OT><<<(unsigned)nblocks, kF8Threads, 0, s>>>(g);
    else
        k_int8_decode_t<OT><<<(unsigned)nblocks, kI8Threads, 0, s>>>(g);
}

template <typename OT>
static void launch_int8_decode_tf(const TFGeom &g, dim3 grid, cudaStream_t s) {
    k_int8_decode_timefirst<OT><<<grid, kTFThreads, 0, s>>>(g);
}

template <typename S>
static void launch_int8_encode_t(const I8Geom &g, uint64_t nblocks, bool fast,
                                 cudaStream_t s) {
    if (fast)
        k_int8_encode_t64<S><<<(unsigned)nblocks, kF8Threads, 0, s>>>(g);
    else
        k_int8_encode_t<S><<<(unsigned)nblocks, kI8Threads, 0, s>>>(g);
}

// Alignment the int8 decoders require of `out`: float32 keeps its 8 / 4
// bytes; the 16-bit types need 8.  0: not a decoder output type.
static int int8_out_align(int32_t out_dtype, int f32_align) {
    const int esize = out_elem_nbytes(out_dtype);
    return esize == 4 ? f32_align : esize == 2 ? 8 : 0;
}

}  // namespace bb

using namespace bb;

extern "C" int bb_decode_int8_transposed_typed(
    const void *src, const int64_t *unit_offset, int64_t nunit, int64_t nrow,
    int64_t ncol, int32_t item_nbytes, const int64_t *col_begin,
    const int64_t *col_end, const int64_t *out_col0, int32_t out_dtype,
    void *out, void *stream) {
    if (!src || !unit_offset || !col_begin || !col_end || !out_col0 || !out)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    const int align = int8_out_align(out_dtype, 8);
    if (align == 0)
        return set_error(BB_ERR_ARGUMENT,
                         "out_dtype must be BB_F32, BB_F16 or BB_BF16");
    if (!aligned(out, align))
        return set_error(BB_ERR_ALIGNMENT, "out must be %d-byte aligned",
                         align);
    I8Geom g;
    uint64_t nblocks;
    // Fast tile kernel: rows paired into float4-equivalent (complex) /
    // float2-equivalent stores.
    const bool fast = nrow % 2 == 0
        && aligned(out, 4 * out_elem_nbytes(out_dtype));
    int rc = fill_geom(g, nunit, nrow, ncol, item_nbytes, nblocks, fast);
    if (rc != BB_OK) return rc;
    if (nblocks == 0) return BB_OK;
    g.src = (const uint8_t *)src;
    g.unit_offset = (const long long *)unit_offset;
    g.col_begin = (const long long *)col_begin;
    g.col_end = (const long long *)col_end;
    g.out_col0 = (const long long *)out_col0;
    g.out = out;
    g.in = nullptr;
    cudaStream_t s = as_stream(stream);
    if (out_dtype == BB_F16) launch_int8_decode_t<F16>(g, nblocks, fast, s);
    else if (out_dtype == BB_BF16) launch_int8_decode_t<BF16>(g, nblocks, fast, s);
    else launch_int8_decode_t<float>(g, nblocks, fast, s);
    BB_CHECK_LAUNCH("bb_decode_int8_transposed launch");
    return BB_OK;
}

extern "C" int bb_decode_int8_transposed(
    const void *src, const int64_t *unit_offset, int64_t nunit, int64_t nrow,
    int64_t ncol, int32_t item_nbytes, const int64_t *col_begin,
    const int64_t *col_end, const int64_t *out_col0, float *out,
    void *stream) {
    return bb_decode_int8_transposed_typed(src, unit_offset, nunit, nrow, ncol,
                                           item_nbytes, col_begin, col_end,
                                           out_col0, BB_F32, out, stream);
}

extern "C" int bb_encode_int8_transposed_typed(
    const void *in, int32_t in_dtype, void *dst, const int64_t *unit_offset,
    int64_t nunit, int64_t nrow, int64_t ncol, int32_t item_nbytes,
    void *stream) {
    if (!in || !dst || !unit_offset)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    const int in_align = in_vec_align(in_dtype);
    if (in_align == 0)
        return set_error(BB_ERR_ARGUMENT,
                         "in_dtype must be BB_F32, BB_F64, BB_F16 or BB_BF16");
    I8Geom g;
    uint64_t nblocks;
    const bool fast = nrow % 2 == 0 && aligned(in, in_align);
    int rc = fill_geom(g, nunit, nrow, ncol, item_nbytes, nblocks, fast);
    if (rc != BB_OK) return rc;
    if (nblocks == 0) return BB_OK;
    g.src = (const uint8_t *)dst;
    g.unit_offset = (const long long *)unit_offset;
    g.col_begin = g.col_end = g.out_col0 = nullptr;
    g.out = nullptr;
    g.in = in;
    cudaStream_t s = as_stream(stream);
    if (in_dtype == BB_F32) launch_int8_encode_t<float>(g, nblocks, fast, s);
    else if (in_dtype == BB_F64) launch_int8_encode_t<double>(g, nblocks, fast, s);
    else if (in_dtype == BB_F16) launch_int8_encode_t<F16>(g, nblocks, fast, s);
    else launch_int8_encode_t<BF16>(g, nblocks, fast, s);
    BB_CHECK_LAUNCH("bb_encode_int8_transposed launch");
    return BB_OK;
}

extern "C" int bb_encode_int8_transposed(
    const void *in, int32_t in_dtype, void *dst, const int64_t *unit_offset,
    int64_t nunit, int64_t nrow, int64_t ncol, int32_t item_nbytes,
    void *stream) {
    if (in_dtype != BB_F32 && in_dtype != BB_F64)
        return set_error(BB_ERR_ARGUMENT, "in_dtype must be BB_F32 or BB_F64");
    return bb_encode_int8_transposed_typed(in, in_dtype, dst, unit_offset,
                                           nunit, nrow, ncol, item_nbytes,
                                           stream);
}

extern "C" int bb_decode_int8_timefirst_typed(
    const void *src, const int64_t *unit_offset, int64_t nunit,
    int64_t nsample, int32_t nchan, int32_t npol, int32_t item_nbytes,
    const int64_t *t_begin, const int64_t *t_end, const int64_t *out_t0,
    int32_t out_dtype, void *out, void *stream) {
    if (!src || !unit_offset || !t_begin || !t_end || !out_t0 || !out)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    const int align = int8_out_align(out_dtype, 4);
    if (align == 0)
        return set_error(BB_ERR_ARGUMENT,
                         "out_dtype must be BB_F32, BB_F16 or BB_BF16");
    if (!aligned(out, align))
        return set_error(BB_ERR_ALIGNMENT, "out must be %d-byte aligned",
                         align);
    TFGeom g;
    if (const char *msg = tf_fill_geom(
            g, nunit, nsample, nchan, npol, item_nbytes,
            aligned(out, 4 * out_elem_nbytes(out_dtype))))
        return set_error(BB_ERR_ARGUMENT, "%s", msg);
    if (nunit == 0) return BB_OK;
    g.src = (const uint8_t *)src;
    g.unit_offset = (const long long *)unit_offset;
    g.t_begin = (const long long *)t_begin;
    g.t_end = (const long long *)t_end;
    g.out_t0 = (const long long *)out_t0;
    g.out = out;
    g.in = nullptr;
    const uint32_t per = kTFThreads * kTFUnroll;
    dim3 grid((g.items_per_unit + per - 1) / per, (unsigned)nunit);
    cudaStream_t s = as_stream(stream);
    if (out_dtype == BB_F16) launch_int8_decode_tf<F16>(g, grid, s);
    else if (out_dtype == BB_BF16) launch_int8_decode_tf<BF16>(g, grid, s);
    else launch_int8_decode_tf<float>(g, grid, s);
    BB_CHECK_LAUNCH("bb_decode_int8_timefirst launch");
    return BB_OK;
}

extern "C" int bb_decode_int8_timefirst(
    const void *src, const int64_t *unit_offset, int64_t nunit,
    int64_t nsample, int32_t nchan, int32_t npol, int32_t item_nbytes,
    const int64_t *t_begin, const int64_t *t_end, const int64_t *out_t0,
    float *out, void *stream) {
    return bb_decode_int8_timefirst_typed(src, unit_offset, nunit, nsample,
                                          nchan, npol, item_nbytes, t_begin,
                                          t_end, out_t0, BB_F32, out, stream);
}

extern "C" int bb_encode_int8_timefirst_typed(
    const void *in, int32_t in_dtype, void *dst, const int64_t *unit_offset,
    int64_t nunit, int64_t nsample, int32_t nchan, int32_t npol,
    int32_t item_nbytes, void *stream) {
    if (!in || !dst || !unit_offset)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    const int in_align = in_vec_align(in_dtype);
    if (in_align == 0)
        return set_error(BB_ERR_ARGUMENT,
                         "in_dtype must be BB_F32, BB_F64, BB_F16 or BB_BF16");
    TFGeom g;
    if (const char *msg = tf_fill_geom(g, nunit, nsample, nchan, npol,
                                       item_nbytes, aligned(in, in_align)))
        return set_error(BB_ERR_ARGUMENT, "%s", msg);
    if (nunit == 0) return BB_OK;
    g.src = (const uint8_t *)dst;
    g.unit_offset = (const long long *)unit_offset;
    g.t_begin = g.t_end = g.out_t0 = nullptr;
    g.out = nullptr;
    g.in = in;
    const uint32_t per = kTFThreads * kTFUnroll;
    dim3 grid((g.items_per_unit + per - 1) / per, (unsigned)nunit);
    cudaStream_t s = as_stream(stream);
    if (in_dtype == BB_F32)
        k_int8_encode_timefirst<float><<<grid, kTFThreads, 0, s>>>(g);
    else if (in_dtype == BB_F64)
        k_int8_encode_timefirst<double><<<grid, kTFThreads, 0, s>>>(g);
    else if (in_dtype == BB_F16)
        k_int8_encode_timefirst<F16><<<grid, kTFThreads, 0, s>>>(g);
    else
        k_int8_encode_timefirst<BF16><<<grid, kTFThreads, 0, s>>>(g);
    BB_CHECK_LAUNCH("bb_encode_int8_timefirst launch");
    return BB_OK;
}

extern "C" int bb_encode_int8_timefirst(
    const void *in, int32_t in_dtype, void *dst, const int64_t *unit_offset,
    int64_t nunit, int64_t nsample, int32_t nchan, int32_t npol,
    int32_t item_nbytes, void *stream) {
    if (in_dtype != BB_F32 && in_dtype != BB_F64)
        return set_error(BB_ERR_ARGUMENT, "in_dtype must be BB_F32 or BB_F64");
    return bb_encode_int8_timefirst_typed(in, in_dtype, dst, unit_offset,
                                          nunit, nsample, nchan, npol,
                                          item_nbytes, stream);
}
