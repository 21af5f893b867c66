// Mark 4 decode/encode kernels and C entry points (sm_100a).
#include <string>
#include <vector>
#include "bb_runtime.cuh"
#include "bb_bitfield.cuh"      // DecodeLut
#include "bb_mark4_plan.h"

namespace bb {

constexpr int kM4Block = 256;
// one-shot grid, ~64 KiB of output per CTA (see bb_bitfield.cu)
// Items per thread, measured per kernel (profiles/README.md): the FAST decode
// wants 4 (16 float4 per thread; 6.43 vs 6.14 / 5.65 TB/s with 2 / 1), the
// WARP decode 2 chunks (+1.5 % over 4), the FAST encode 1 (6.86 vs 6.66 /
// 6.41 with 2 / 4), the HALF encode 4.
constexpr int kM4UnrollFast = 4, kM4UnrollVec = 16, kM4UnrollScalar = 16,
    kM4UnrollWarp = 2, kM4UnrollEncFast = 1, kM4UnrollHalf = 4;

static inline unsigned m4_grid(uint32_t nitems, int unroll) {
    uint64_t per = (uint64_t)kM4Block * unroll;
    return (unsigned)((nitems + per - 1) / per);
}

template <int MODE, typename OT>
__global__ void __launch_bounds__(kM4Block) k_mark4_decode(const M4Geom p) {
    // pair LUT over the raw code (sign | magnitude << 1), see DecodeLut<2>
    __shared__ __align__(16) float lut[DecodeLut<2>::kFloats];
    if (MODE == M4_FAST || MODE == M4_WARP) {
        if (threadIdx.x < DecodeLut<2>::kFloats) {
            int entry = threadIdx.x >> 1, which = threadIdx.x & 1;
            int code = which ? (entry >> 2) : (entry & 3);
            lut[threadIdx.x] = p.levels[2 * (code & 1) + (code >> 1)];
        }
        __syncthreads();
    }
    constexpr int U = MODE == M4_FAST ? kM4UnrollFast
        : MODE == M4_WARP ? kM4UnrollWarp
        : MODE == M4_GENERIC_VEC ? kM4UnrollVec : kM4UnrollScalar;
    const uint32_t item0 = blockIdx.x * (kM4Block * U) + threadIdx.x;
    if (MODE == M4_WARP) {
        const uint32_t lane = threadIdx.x & 31u;
        const M4Lane lc = m4w_lane(p, p.pos, lane);
        const float lv[4] = {p.levels[0], p.levels[1], p.levels[2],
                             p.levels[3]};
        uint32_t w[U];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t item = item0 + u * kM4Block;
            ok[u] = item < p.nitems && m4w_load(p, item >> 5, lane, w[u]);
        }
        if (p.std4) {                              // launch uniform
            const uint32_t row = m4s_row(p, lane);
            uint32_t ssrc[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) ssrc[j] = m4s_src_lane(p, lane + 32u * j);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t item = item0 + u * kM4Block;
                if (item >= p.nitems) break;       // warp uniform
                const unsigned okmask = __ballot_sync(0xffffffffu, ok[u]);
                if (m4w_interior(p, item >> 5)) {
                    OT *chunk_out = m4w_chunk_out<OT>(p, item >> 5);
                    const uint32_t r = m4_reorder32(w[u]);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t rs = __shfl_sync(0xffffffffu, r, ssrc[j]);
                        m4s_emit_fast(p, lut, chunk_out, lane + 32u * j, row,
                                      rs, (okmask >> ssrc[j]) & 1u);
                    }
                    continue;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t q = lane + 32u * j;
                    const uint32_t src = m4w_src_lane(p, lc, q);
                    const uint32_t ws = __shfl_sync(0xffffffffu, w[u], src);
                    m4w_emit<OT>(p, lc, lv, item >> 5, q, ws, (okmask >> src) & 1u);
                }
            }
            return;
        }
        uint32_t srcl[4];                          // loop-invariant per lane
#pragma unroll
        for (int j = 0; j < 4; ++j) srcl[j] = m4w_src_lane(p, lc, lane + 32u * j);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t item = item0 + u * kM4Block;
            if (item >= p.nitems) break;           // warp uniform
            const unsigned okmask = __ballot_sync(0xffffffffu, ok[u]);
            if (m4w_interior(p, item >> 5)) {      // warp uniform
                OT *chunk_out = m4w_chunk_out<OT>(p, item >> 5);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t ws = __shfl_sync(0xffffffffu, w[u], srcl[j]);
                    m4w_emit_fast(p, lc, lut, chunk_out, lane + 32u * j, ws,
                                  (okmask >> srcl[j]) & 1u);
                }
                continue;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t q = lane + 32u * j;
                const uint32_t src = m4w_src_lane(p, lc, q);
                const uint32_t ws = __shfl_sync(0xffffffffu, w[u], src);
                m4w_emit<OT>(p, lc, lv, item >> 5, q, ws, (okmask >> src) & 1u);
            }
        }
        return;
    }
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
        const uint32_t item = item0 + u * kM4Block;
        if (item >= p.nitems) break;
        if (MODE == M4_FAST) m4_dec_fast<OT>(p, lut, item);
        else if (MODE == M4_GENERIC_VEC) m4_dec_generic<true, OT>(p, item);
        else m4_dec_generic<false, OT>(p, item);
    }
}

template <typename S, int MODE>
__global__ void __launch_bounds__(kM4Block)
k_mark4_encode(const M4Geom p, const QuantConsts<arith_t<S>> c) {
    constexpr int U = kM4UnrollEncFast;
    const uint32_t item0 = blockIdx.x * (kM4Block * U) + threadIdx.x;
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
        const uint32_t item = item0 + u * kM4Block;
        if (item >= p.nitems) break;
        if (MODE == M4_FAST) m4_enc_fast<S>(p, c, item);
        else m4_enc_generic<S>(p, c, item);
    }
}

// HALF encode, one kernel per track-word size: the bit masks of a thread are
// built once (they only depend on the layout and the parity of the item).
template <typename S, int W>
__global__ void __launch_bounds__(kM4Block)
k_mark4_encode_half(const M4Geom p, const QuantConsts<arith_t<S>> c) {
    constexpr int U = kM4UnrollHalf;
    const uint32_t item0 = blockIdx.x * (kM4Block * U) + threadIdx.x;
    // kM4Block is even: every item of this thread has the parity of item0
    const M4HalfMasks mk = m4_half_masks<W>(p, p.pos, item0 & 1u);
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
        const uint32_t item = item0 + u * kM4Block;
        if (item >= p.nitems) break;
        m4_enc_half_w<S, W>(p, mk, c, item);
    }
}

template <typename OT>
static int run_decode(const std::vector<M4Launch> &launches, cudaStream_t s) {
    for (const M4Launch &l : launches) {
        const uint32_t n = l.g.nitems;
        if (l.mode == M4_FAST)
            k_mark4_decode<M4_FAST, OT>
                <<<m4_grid(n, kM4UnrollFast), kM4Block, 0, s>>>(l.g);
        else if (l.mode == M4_WARP)
            k_mark4_decode<M4_WARP, OT>
                <<<m4_grid(n, kM4UnrollWarp), kM4Block, 0, s>>>(l.g);
        else if (l.mode == M4_GENERIC_VEC)
            k_mark4_decode<M4_GENERIC_VEC, OT>
                <<<m4_grid(n, kM4UnrollVec), kM4Block, 0, s>>>(l.g);
        else
            k_mark4_decode<M4_GENERIC_SCALAR, OT>
                <<<m4_grid(n, kM4UnrollScalar), kM4Block, 0, s>>>(l.g);
        BB_CHECK_LAUNCH("bb_mark4_decode launch");
    }
    return BB_OK;
}

template <typename S>
static int run_encode(const std::vector<M4Launch> &launches, cudaStream_t s) {
    using T = arith_t<S>;
    static const QuantConsts<T> consts = make_quant_consts<T>();
    for (const M4Launch &l : launches) {
        unsigned grid = m4_grid(l.g.nitems, l.mode == M4_HALF
                                ? kM4UnrollHalf : kM4UnrollEncFast);
        if (l.mode == M4_FAST)
            k_mark4_encode<S, M4_FAST><<<grid, kM4Block, 0, s>>>(l.g, consts);
        else if (l.mode == M4_HALF && l.g.wordbytes == 8)
            k_mark4_encode_half<S, 8><<<grid, kM4Block, 0, s>>>(l.g, consts);
        else if (l.mode == M4_HALF && l.g.wordbytes == 4)
            k_mark4_encode_half<S, 4><<<grid, kM4Block, 0, s>>>(l.g, consts);
        else if (l.mode == M4_HALF)
            k_mark4_encode_half<S, 2><<<grid, kM4Block, 0, s>>>(l.g, consts);
        else
            k_mark4_encode<S, M4_GENERIC_SCALAR>
                <<<grid, kM4Block, 0, s>>>(l.g, consts);
        BB_CHECK_LAUNCH("bb_mark4_encode launch");
    }
    return BB_OK;
}

}  // namespace bb

using namespace bb;

extern "C" int bb_mark4_decode_typed(
    const void *src, const int64_t *unit_offset, int64_t nframe, int32_t nchan,
    int32_t fanout, int32_t ft, const float *levels_host, float fill_value,
    int64_t sample_start, int64_t nsample, int32_t out_dtype, void *out,
    void *stream) {
    if (!src || !unit_offset || !out || !levels_host)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    const int esize = out_elem_nbytes(out_dtype);
    if (esize == 0)
        return set_error(BB_ERR_ARGUMENT,
                         "out_dtype must be BB_F32, BB_F16 or BB_BF16");
    if (!aligned(out, 4 * esize) || !aligned(src, 8))
        return set_error(BB_ERR_ALIGNMENT,
                         "out must be %d-byte and src 8-byte aligned",
                         4 * esize);
    std::vector<M4Launch> launches;
    std::string err;
    if (!plan_m4_frames(false, src, unit_offset, nframe, nchan, fanout, ft,
                        levels_host, fill_value, sample_start, nsample, out,
                        nullptr, launches, err))
        return set_error(err.rfind("no Mark 4 codec", 0) == 0
                         ? BB_ERR_UNSUPPORTED : BB_ERR_ARGUMENT, "%s",
                         err.c_str());
    cudaStream_t s = as_stream(stream);
    if (out_dtype == BB_F16) return run_decode<F16>(launches, s);
    if (out_dtype == BB_BF16) return run_decode<BF16>(launches, s);
    return run_decode<float>(launches, s);
}

extern "C" int bb_mark4_decode(
    const void *src, const int64_t *unit_offset, int64_t nframe, int32_t nchan,
    int32_t fanout, int32_t ft, const float *levels_host, float fill_value,
    int64_t sample_start, int64_t nsample, float *out, void *stream) {
    return bb_mark4_decode_typed(src, unit_offset, nframe, nchan, fanout, ft,
                                 levels_host, fill_value, sample_start,
                                 nsample, BB_F32, out, stream);
}

extern "C" int bb_mark4_encode_typed(
    const void *in, int32_t in_dtype, void *dst, const int64_t *unit_offset,
    int64_t nframe, int32_t nchan, int32_t fanout, int32_t ft, void *stream) {
    if (!in || !dst || !unit_offset)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    const int in_align = in_vec_align(in_dtype);
    if (in_align == 0)
        return set_error(BB_ERR_ARGUMENT,
                         "in_dtype must be BB_F32, BB_F64, BB_F16 or BB_BF16");
    if (!aligned(in, in_align) || !aligned(dst, 8))
        return set_error(BB_ERR_ALIGNMENT,
                         "in must be %d-byte and dst 8-byte aligned",
                         in_align);
    std::vector<M4Launch> launches;
    std::string err;
    if (!plan_m4_frames(true, dst, unit_offset, nframe, nchan, fanout, ft,
                        nullptr, 0.f, 0, nframe * 20000ll * fanout, nullptr, in,
                        launches, err, in_align))
        return set_error(err.rfind("no Mark 4 codec", 0) == 0
                         ? BB_ERR_UNSUPPORTED : BB_ERR_ARGUMENT, "%s",
                         err.c_str());
    cudaStream_t s = as_stream(stream);
    if (in_dtype == BB_F32) return run_encode<float>(launches, s);
    if (in_dtype == BB_F64) return run_encode<double>(launches, s);
    if (in_dtype == BB_F16) return run_encode<F16>(launches, s);
    return run_encode<BF16>(launches, s);
}

extern "C" int bb_mark4_encode(
    const void *in, int32_t in_dtype, void *dst, const int64_t *unit_offset,
    int64_t nframe, int32_t nchan, int32_t fanout, int32_t ft, void *stream) {
    if (in_dtype != BB_F32 && in_dtype != BB_F64)
        return set_error(BB_ERR_ARGUMENT, "in_dtype must be BB_F32 or BB_F64");
    return bb_mark4_encode_typed(in, in_dtype, dst, unit_offset, nframe, nchan,
                                 fanout, ft, stream);
}

extern "C" int bb_mark4_decode_words(
    const void *words, int64_t nword, int32_t nchan, int32_t fanout,
    int32_t ft, const float *levels_host, float *out, void *stream) {
    if (!words || !out || !levels_host)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    if (!aligned(out, 16) || !aligned(words, 8))
        return set_error(BB_ERR_ALIGNMENT,
                         "out must be 16-byte and words 8-byte aligned");
    std::vector<M4Launch> launches;
    std::string err;
    if (!plan_m4_words(false, words, nword, nchan, fanout, ft, levels_host,
                       out, nullptr, launches, err))
        return set_error(err.rfind("no Mark 4 codec", 0) == 0
                         ? BB_ERR_UNSUPPORTED : BB_ERR_ARGUMENT, "%s",
                         err.c_str());
    return run_decode<float>(launches, as_stream(stream));
}

extern "C" int bb_mark4_encode_words(
    const void *in, int32_t in_dtype, void *words, int64_t nword,
    int32_t nchan, int32_t fanout, int32_t ft, void *stream) {
    if (!in || !words)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    if (!aligned(in, 16) || !aligned(words, 8))
        return set_error(BB_ERR_ALIGNMENT,
                         "in must be 16-byte and words 8-byte aligned");
    std::vector<M4Launch> launches;
    std::string err;
    if (!plan_m4_words(true, words, nword, nchan, fanout, ft, nullptr, nullptr,
                       in, launches, err))
        return set_error(err.rfind("no Mark 4 codec", 0) == 0
                         ? BB_ERR_UNSUPPORTED : BB_ERR_ARGUMENT, "%s",
                         err.c_str());
    if (in_dtype == BB_F32) return run_encode<float>(launches, as_stream(stream));
    if (in_dtype == BB_F64) return run_encode<double>(launches, as_stream(stream));
    return set_error(BB_ERR_ARGUMENT, "in_dtype must be BB_F32 or BB_F64");
}
