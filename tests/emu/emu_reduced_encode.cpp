// CPU emulation of the float16 / bfloat16 encode paths — TEST INFRASTRUCTURE
// ONLY (see emu_bitfield.cpp).  The four `_typed` encoders of the C ABI run
// the same per-thread bodies with the input storage type S (float, double,
// F16, BF16), with the library's argument and alignment checks, so the
// widening on load, the planner's choices and the edge paths of the 16-bit
// encoders are checked on the CPU.  Never loaded by baseband_b200.
#include <cstdint>
#include <string>
#include <vector>
#include "../../baseband_b200/csrc/bb_bitfield_plan.h"
#include "../../baseband_b200/csrc/bb_mark4_plan.h"
#include "../../baseband_b200/csrc/bb_int8.cuh"
#include "../../include/baseband_b200.h"

using namespace bb;

static std::string g_err_enc;

// bytes of one four-value input load; 0: not an encoder input type
static int in_align_of(int32_t in_dtype) {
    return (in_dtype == BB_F32 || in_dtype == BB_F64) ? 16
        : (in_dtype == BB_F16 || in_dtype == BB_BF16) ? 8 : 0;
}

static bool is_aligned(const void *p, int a) {
    return (reinterpret_cast<uintptr_t>(p) % (uintptr_t)a) == 0;
}

// ------------------------------------------------------------- bit field
template <typename S, int BPS, int QUANT>
static void enc_bitfield(const std::vector<EncLaunch> &launches) {
    using T = arith_t<S>;
    const QuantConsts<T> c = make_quant_consts<T>();
    for (const EncLaunch &l : launches) {
        if (l.mode == MODE_ROWWORD4 || l.mode == MODE_ROWWORD2) {
            std::vector<uint32_t> buf(32 * 32);
            for (uint32_t chunk = 0; chunk < l.g.nitems / 32; ++chunk) {
                for (uint32_t lane = 0; lane < 32; ++lane) {
                    if (l.mode == MODE_ROWWORD4)
                        rw_stage<S, BPS, QUANT, 4>(l.g, c, chunk, lane, buf.data());
                    else
                        rw_stage<S, BPS, QUANT, 2>(l.g, c, chunk, lane, buf.data());
                }
                for (uint32_t lane = 0; lane < 32; ++lane) {
                    if (l.mode == MODE_ROWWORD4)
                        rw_emit<BPS, 4>(l.g, chunk, lane, buf.data());
                    else
                        rw_emit<BPS, 2>(l.g, chunk, lane, buf.data());
                }
            }
            continue;
        }
        for (uint32_t item = 0; item < l.g.nitems; ++item) {
            if (l.mode == MODE_ROWGROUP4) enc_rowgroup<S, BPS, QUANT, 4>(l.g, c, item);
            else if (l.mode == MODE_ROWGROUP2) enc_rowgroup<S, BPS, QUANT, 2>(l.g, c, item);
            else if (l.mode == MODE_RUN) enc_word<S, BPS, QUANT, true>(l.g, c, item);
            else if (l.mode == MODE_RUNQ) {
                EncQuadItem<T> it;
                enc_quad_fetch<S>(l.g, item, it);
                enc_quad_emit<T, QUANT>(c, it);
            } else enc_word<S, BPS, QUANT, false>(l.g, c, item);
        }
    }
}

template <typename S>
static int enc_bitfield_dispatch(int bps, int q,
                                 const std::vector<EncLaunch> &l) {
    if (q == BB_QUANT_OFFSET_BINARY) {
        if (bps == 1) return enc_bitfield<S, 1, QUANT_OFFSET>(l), 0;
        if (bps == 2) return enc_bitfield<S, 2, QUANT_OFFSET>(l), 0;
        if (bps == 4) return enc_bitfield<S, 4, QUANT_OFFSET>(l), 0;
        if (bps == 8) return enc_bitfield<S, 8, QUANT_OFFSET>(l), 0;
    } else if (q == BB_QUANT_MARK5B) {
        if (bps == 1) return enc_bitfield<S, 1, QUANT_MARK5B>(l), 0;
        if (bps == 2) return enc_bitfield<S, 2, QUANT_MARK5B>(l), 0;
    } else if (q == BB_QUANT_SINT) {
        if (bps == 4) return enc_bitfield<S, 4, QUANT_SINT>(l), 0;
        if (bps == 8) return enc_bitfield<S, 8, QUANT_SINT>(l), 0;
    }
    return BB_ERR_UNSUPPORTED;
}

// ---------------------------------------------------------------- Mark 4
template <typename S>
static void enc_mark4(const std::vector<M4Launch> &launches) {
    const QuantConsts<arith_t<S>> c = make_quant_consts<arith_t<S>>();
    for (const M4Launch &l : launches)
        for (uint32_t item = 0; item < l.g.nitems; ++item) {
            if (l.mode == M4_FAST) m4_enc_fast<S>(l.g, c, item);
            else if (l.mode == M4_HALF) m4_enc_half<S>(l.g, l.g.pos, c, item);
            else m4_enc_generic<S>(l.g, c, item);
        }
}

// ------------------------------------------------------------------ int8
template <typename S>
static void enc_int8_t(const I8Geom &g, uint64_t nblocks, bool fast) {
    if (fast) {
        std::vector<uint32_t> tile64(kF8SmemWords);
        for (uint64_t b = 0; b < nblocks; ++b) {
            for (uint32_t t = 0; t < kF8Threads; ++t)
                f8_enc_load<S>(g, tile64.data(), (uint32_t)b, t);
            for (uint32_t t = 0; t < kF8Threads; ++t)
                f8_enc_store(g, tile64.data(), (uint32_t)b, t);
        }
        return;
    }
    alignas(16) uint8_t tile[kI8SmemBytes];
    for (uint64_t b = 0; b < nblocks; ++b) {
        for (uint32_t t = 0; t < kI8Threads; ++t) i8_enc_load<S>(g, tile, (uint32_t)b, t);
        for (uint32_t t = 0; t < kI8Threads; ++t) i8_enc_store(g, tile, (uint32_t)b, t);
    }
}

extern "C" {

const char *emu_reduced_encode_error(void) { return g_err_enc.c_str(); }

int bb_encode_bitfield_typed(const void *in, int32_t in_dtype, void *dst,
                             const int64_t *unit_offset, int64_t nset,
                             int32_t nthread, int64_t payload_nbytes,
                             int32_t bps, int32_t nelem, int32_t quantiser,
                             void *stream) {
    const int a = in_align_of(in_dtype);
    if (!in || !dst || !unit_offset || a == 0) return BB_ERR_ARGUMENT;
    if (!is_aligned(in, a) || !is_aligned(dst, 4)) return BB_ERR_ALIGNMENT;
    std::vector<EncLaunch> l;
    if (!plan_encode(in, dst, unit_offset, nset, nthread, payload_nbytes, bps,
                     nelem, l, g_err_enc))
        return BB_ERR_ARGUMENT;
    if (in_dtype == BB_F32) return enc_bitfield_dispatch<float>(bps, quantiser, l);
    if (in_dtype == BB_F64) return enc_bitfield_dispatch<double>(bps, quantiser, l);
    if (in_dtype == BB_F16) return enc_bitfield_dispatch<F16>(bps, quantiser, l);
    return enc_bitfield_dispatch<BF16>(bps, quantiser, l);
}

int bb_mark4_encode_typed(const void *in, int32_t in_dtype, void *dst,
                          const int64_t *unit_offset, int64_t nframe,
                          int32_t nchan, int32_t fanout, int32_t ft,
                          void *stream) {
    const int a = in_align_of(in_dtype);
    if (!in || !dst || !unit_offset || a == 0) return BB_ERR_ARGUMENT;
    if (!is_aligned(in, a) || !is_aligned(dst, 8)) return BB_ERR_ALIGNMENT;
    std::vector<M4Launch> l;
    if (!plan_m4_frames(true, dst, unit_offset, nframe, nchan, fanout, ft,
                        nullptr, 0.f, 0, nframe * 20000ll * fanout, nullptr,
                        in, l, g_err_enc, (uintptr_t)a))
        return BB_ERR_ARGUMENT;
    if (in_dtype == BB_F32) enc_mark4<float>(l);
    else if (in_dtype == BB_F64) enc_mark4<double>(l);
    else if (in_dtype == BB_F16) enc_mark4<F16>(l);
    else enc_mark4<BF16>(l);
    return 0;
}

int bb_encode_int8_transposed_typed(const void *in, int32_t in_dtype,
                                    void *dst, const int64_t *unit_offset,
                                    int64_t nunit, int64_t nrow, int64_t ncol,
                                    int32_t item_nbytes, void *stream) {
    const int a = in_align_of(in_dtype);
    if (!in || !dst || !unit_offset || a == 0) return BB_ERR_ARGUMENT;
    if (item_nbytes != 1 && item_nbytes != 2) return BB_ERR_ARGUMENT;
    const bool fast = nrow % 2 == 0 && is_aligned(in, a);
    I8Geom g;
    g.nunit = (uint32_t)nunit; g.nrow = (uint32_t)nrow; g.ncol = (uint32_t)ncol;
    g.ib = item_nbytes;
    const int rows = fast ? kF8Rows : kI8Rows;
    g.tiles_r = (uint32_t)((nrow + rows - 1) / rows);
    const uint32_t tc = (fast ? kF8Words * 4 : kI8RowBytes) / item_nbytes;
    g.tiles_c = (uint32_t)((ncol + tc - 1) / tc);
    g.group = 16 < g.tiles_c ? 16 : g.tiles_c;
    if (g.group < 1) g.group = 1;
    g.knock = 0;
    const uint64_t nblocks = (uint64_t)nunit * g.tiles_r * g.tiles_c;
    g.src = (const uint8_t *)dst;
    g.unit_offset = (const long long *)unit_offset;
    g.col_begin = g.col_end = g.out_col0 = nullptr;
    g.out = nullptr; g.in = in;
    if (in_dtype == BB_F32) enc_int8_t<float>(g, nblocks, fast);
    else if (in_dtype == BB_F64) enc_int8_t<double>(g, nblocks, fast);
    else if (in_dtype == BB_F16) enc_int8_t<F16>(g, nblocks, fast);
    else enc_int8_t<BF16>(g, nblocks, fast);
    return 0;
}

int bb_encode_int8_timefirst_typed(const void *in, int32_t in_dtype,
                                   void *dst, const int64_t *unit_offset,
                                   int64_t nunit, int64_t nsample,
                                   int32_t nchan, int32_t npol,
                                   int32_t item_nbytes, void *stream) {
    const int a = in_align_of(in_dtype);
    if (!in || !dst || !unit_offset || a == 0) return BB_ERR_ARGUMENT;
    TFGeom g;
    if (tf_fill_geom(g, nunit, nsample, nchan, npol, item_nbytes,
                     is_aligned(in, a)))
        return BB_ERR_ARGUMENT;
    g.src = (const uint8_t *)dst;
    g.unit_offset = (const long long *)unit_offset;
    g.t_begin = g.t_end = g.out_t0 = nullptr;
    g.out = nullptr; g.in = in;
    for (uint32_t u = 0; u < g.nunit; ++u)
        for (uint32_t i = 0; i < g.items_per_unit; ++i) {
            if (in_dtype == BB_F32) tf_encode<float>(g, u, i);
            else if (in_dtype == BB_F64) tf_encode<double>(g, u, i);
            else if (in_dtype == BB_F16) tf_encode<F16>(g, u, i);
            else tf_encode<BF16>(g, u, i);
        }
    return 0;
}

// The host widening the emulation loads 16-bit input with (bb_common.cuh):
// n patterns of half (brain = 0) or bfloat16 (brain = 1) -> float32.
void emu_widen_half(const uint16_t *in, int64_t n, int32_t brain,
                    float *out) {
    for (int64_t i = 0; i < n; ++i)
        out[i] = brain ? widen(BF16{in[i]}) : widen(F16{in[i]});
}

}  // extern "C"
