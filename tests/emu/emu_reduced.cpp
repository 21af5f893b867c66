// CPU emulation of the float16 / bfloat16 decode paths — TEST INFRASTRUCTURE
// ONLY (see emu_bitfield.cpp).  The `_typed` entry points of the C ABI run
// the same per-thread bodies with the output type OT (float, F16, BF16), so
// the planner modes and the edge / fill logic of the 16-bit stores are
// checked on the CPU.  Never loaded by baseband_b200.
#include <cstring>
#include <string>
#include <vector>
#include "../../baseband_b200/csrc/bb_bitfield_plan.h"
#include "../../baseband_b200/csrc/bb_mark4_plan.h"
#include "../../baseband_b200/csrc/bb_int8.cuh"
#include "../../include/baseband_b200.h"

using namespace bb;

static std::string g_err_typed;

// ------------------------------------------------------------- bit field
template <int BPS, int CODEC, int G, int NG, typename OT>
static void typed_wordrow(const DecGeom &g, const float *lut) {
    constexpr int TPW = (32 / BPS) / (4 / G);
    constexpr int W = G * NG;
    for (uint32_t chunk = 0; chunk < g.nitems / 32; ++chunk) {
        uint32_t w[32][W], ok[32];
        for (uint32_t lane = 0; lane < 32; ++lane)
            ok[lane] = wrow_load<W>(g, chunk, lane, w[lane]);
        const bool interior = wrow_interior<BPS, G>(g, chunk);
        for (uint32_t lane = 0; lane < 32; ++lane)
            for (int j = 0; j < TPW * NG; ++j) {
                const uint32_t q = lane + 32u * j;
                const uint32_t src = wrow_src_lane<BPS, G, NG>(lane, j);
                const uint32_t grp = q % NG;
                const uint32_t okg = (ok[src] >> (grp * G)) & ((1u << G) - 1u);
                if (interior)
                    wrow_emit_fast<BPS, CODEC, G, NG>(
                        g, lut, wrow_chunk_out<BPS, G, NG, OT>(g, chunk), q,
                        &w[src][grp * G], okg);
                else
                    wrow_emit<BPS, CODEC, G, NG, OT>(g, lut, chunk, lane, j,
                                                     &w[src][grp * G], okg);
            }
    }
}

template <int BPS, int CODEC, int G, int P, bool SEL, typename OT>
static void typed_tile(const DecGeom &g, const float *lut,
                       const float *levels) {
    using T = Tile<BPS, G, P>;
    LevelTable<BPS> lv;
    for (int i = 0; i < (1 << BPS); ++i) lv.v[i] = levels ? levels[i] : 0.f;
    for (uint32_t chunk = 0; chunk < g.nitems / 32; ++chunk) {
        uint32_t wbuf[T::kWords], oks[32];
        bool full = true;
        for (uint32_t lane = 0; lane < 32; ++lane) {
            uint32_t w[T::kNl];
            oks[lane] = tile_load<BPS, G, P>(g, chunk, lane, w);
            full = full && oks[lane] == (1u << T::kNl) - 1u;
            for (int i = 0; i < T::kNl; ++i) wbuf[T::kNl * lane + i] = w[i];
        }
        const bool fast = full && tile_interior<BPS, G, P>(g, chunk);
        for (uint32_t q = 0; q < 32u * T::kStores; ++q) {
            const uint32_t at = ((q >> 2) / T::kTpw) * T::kSlots + (q & 3u) * G;
            if (fast)
                store4(tile_chunk_out<BPS, G, P, OT>(g, chunk) + 4u * q,
                       tile_decode<BPS, CODEC, G, P, SEL>(q, &wbuf[at], lut,
                                                          lv));
            else
                tile_emit<BPS, CODEC, G, P, SEL, OT>(
                    g, lut, lv, chunk, q, &wbuf[at],
                    full ? (1u << G) - 1u : tile_group_ok<BPS, G, P>(oks, q));
        }
    }
}

template <int BPS, int CODEC, typename OT>
static void typed_decode(const std::vector<DecLaunch> &launches,
                         const float *levels) {
    using Lut = DecodeLut<BPS>;
    alignas(16) float lut[Lut::kFloats];
    if (CODEC == CODEC_LEVELS)
        for (int i = 0; i < Lut::kFloats; ++i) lut[i] = Lut::value(levels, i);
    for (const DecLaunch &l : launches) {
        if (l.mode == MODE_WORDRUN) {
            constexpr int F = 8 / BPS;
            for (uint32_t chunk = 0; chunk < l.g.nitems / 32; ++chunk) {
                uint32_t w[32];
                bool ok[32];
                for (uint32_t lane = 0; lane < 32; ++lane)
                    ok[lane] = wr_load(l.g, chunk, lane, w[lane]);
                for (uint32_t lane = 0; lane < 32; ++lane)
                    for (int j = 0; j < F; ++j) {
                        uint32_t src = wr_src_lane<BPS>(lane, j);
                        wr_emit<BPS, CODEC, OT>(l.g, lut, chunk, lane, j,
                                                w[src], ok[src]);
                    }
            }
            continue;
        }
        if (is_tile(l.mode)) {
            if constexpr (BPS == 2 && CODEC == CODEC_LEVELS) {
                const bool g4 = l.mode == MODE_TILE4;
                if (g4 && l.tile_p == 8 && l.sel) typed_tile<BPS, CODEC, 4, 8, true, OT>(l.g, lut, levels);
                else if (g4 && l.tile_p == 8) typed_tile<BPS, CODEC, 4, 8, false, OT>(l.g, lut, levels);
                else if (g4 && l.sel) typed_tile<BPS, CODEC, 4, 4, true, OT>(l.g, lut, levels);
                else if (g4) typed_tile<BPS, CODEC, 4, 4, false, OT>(l.g, lut, levels);
                else if (l.tile_p == 8 && l.sel) typed_tile<BPS, CODEC, 2, 8, true, OT>(l.g, lut, levels);
                else if (l.tile_p == 8) typed_tile<BPS, CODEC, 2, 8, false, OT>(l.g, lut, levels);
                else if (l.sel) typed_tile<BPS, CODEC, 2, 4, true, OT>(l.g, lut, levels);
                else typed_tile<BPS, CODEC, 2, 4, false, OT>(l.g, lut, levels);
            }
            continue;
        }
        if (is_wordrow(l.mode)) {
            if (l.mode == MODE_WORDROW4) typed_wordrow<BPS, CODEC, 4, 1, OT>(l.g, lut);
            else if (l.mode == MODE_WORDROW2) typed_wordrow<BPS, CODEC, 2, 1, OT>(l.g, lut);
            else if (l.mode == MODE_WORDROW4X2) typed_wordrow<BPS, CODEC, 4, 2, OT>(l.g, lut);
            else typed_wordrow<BPS, CODEC, 2, 2, OT>(l.g, lut);
            continue;
        }
        for (uint32_t item = 0; item < l.g.nitems; ++item) {
            if (l.sel && (l.mode == MODE_ROWGROUP4
                          || l.mode == MODE_ROWGROUP2)) {
                if constexpr (BPS <= 2 && CODEC == CODEC_LEVELS) {
                    LevelTable<BPS> lv;
                    for (int i = 0; i < (1 << BPS); ++i) lv.v[i] = levels[i];
                    if (l.mode == MODE_ROWGROUP4) {
                        RowItem<4> it;
                        rowgroup_fetch<BPS, 4>(l.g, item, it);
                        rowgroup_emit<BPS, CODEC, 4, true, OT>(l.g, lut, it, lv);
                    } else {
                        RowItem<2> it;
                        rowgroup_fetch<BPS, 2>(l.g, item, it);
                        rowgroup_emit<BPS, CODEC, 2, true, OT>(l.g, lut, it, lv);
                    }
                }
                continue;
            }
            if (l.mode == MODE_ROWGROUP4) dec_rowgroup<BPS, CODEC, 4, OT>(l.g, lut, item);
            else if (l.mode == MODE_ROWGROUP2) dec_rowgroup<BPS, CODEC, 2, OT>(l.g, lut, item);
            else if (l.mode == MODE_RUN) dec_run<BPS, CODEC, OT>(l.g, lut, item);
            else if (l.mode == MODE_RUNS) dec_runs<BPS, CODEC, OT>(l.g, lut, item);
            else dec_scalar<BPS, CODEC, OT>(l.g, lut, item);
        }
    }
}

template <typename OT>
static int typed_dispatch(int bps, int codec, const float *levels_host,
                          const std::vector<DecLaunch> &l) {
    if (codec == BB_CODEC_LEVELS) {
        if (bps == 1) return typed_decode<1, CODEC_LEVELS, OT>(l, levels_host), 0;
        if (bps == 2) return typed_decode<2, CODEC_LEVELS, OT>(l, levels_host), 0;
        if (bps == 4) return typed_decode<4, CODEC_LEVELS, OT>(l, levels_host), 0;
        if (bps == 8 && affine8_matches(levels_host))
            return typed_decode<8, CODEC_AFFINE8, OT>(l, nullptr), 0;
        if (bps == 8) return typed_decode<8, CODEC_LEVELS, OT>(l, levels_host), 0;
    } else {
        if (bps == 4) return typed_decode<4, CODEC_SINT, OT>(l, nullptr), 0;
        if (bps == 8) return typed_decode<8, CODEC_SINT, OT>(l, nullptr), 0;
    }
    return BB_ERR_UNSUPPORTED;
}

// ---------------------------------------------------------------- Mark 4
template <typename OT>
static void typed_mark4(const std::vector<M4Launch> &launches) {
    for (const M4Launch &l : launches) {
        alignas(16) float lut[DecodeLut<2>::kFloats];
        for (int i = 0; i < DecodeLut<2>::kFloats; ++i) {
            int entry = i >> 1, which = i & 1;
            int code = which ? (entry >> 2) : (entry & 3);
            lut[i] = l.g.levels[2 * (code & 1) + (code >> 1)];
        }
        if (l.mode == M4_WARP) {
            for (uint32_t chunk = 0; chunk < l.g.nitems / 32; ++chunk) {
                uint32_t w[32];
                bool ok[32];
                for (uint32_t lane = 0; lane < 32; ++lane)
                    ok[lane] = m4w_load(l.g, chunk, lane, w[lane]);
                const bool interior = m4w_interior(l.g, chunk);
                for (uint32_t q = 0; q < 128; ++q) {
                    const M4Lane lc = m4w_lane(l.g, l.g.pos, q & 31u);
                    uint32_t src = m4w_src_lane(l.g, lc, q);
                    if (interior && l.g.std4) {
                        const uint32_t ss = m4s_src_lane(l.g, q);
                        m4s_emit_fast(l.g, lut, m4w_chunk_out<OT>(l.g, chunk),
                                      q, m4s_row(l.g, q), m4_reorder32(w[ss]),
                                      ok[ss]);
                    } else if (interior)
                        m4w_emit_fast(l.g, lc, lut,
                                      m4w_chunk_out<OT>(l.g, chunk), q, w[src],
                                      ok[src]);
                    else
                        m4w_emit<OT>(l.g, lc, l.g.levels, chunk, q, w[src],
                                     ok[src]);
                }
            }
            continue;
        }
        for (uint32_t item = 0; item < l.g.nitems; ++item) {
            if (l.mode == M4_FAST) m4_dec_fast<OT>(l.g, lut, item);
            else if (l.mode == M4_GENERIC_VEC) m4_dec_generic<true, OT>(l.g, item);
            else m4_dec_generic<false, OT>(l.g, item);
        }
    }
}

// ------------------------------------------------------------------ int8
template <typename OT>
static void typed_int8_t(const I8Geom &g, uint64_t nblocks, bool fast) {
    if (fast) {
        std::vector<uint32_t> tile64(kF8SmemWords);
        for (uint64_t b = 0; b < nblocks; ++b) {
            for (uint32_t t = 0; t < kF8Threads; ++t)
                f8_dec_load(g, tile64.data(), (uint32_t)b, t);
            for (uint32_t t = 0; t < kF8Threads; ++t)
                f8_dec_store<OT>(g, tile64.data(), (uint32_t)b, t);
        }
        return;
    }
    alignas(16) uint8_t tile[kI8SmemBytes];
    for (uint64_t b = 0; b < nblocks; ++b) {
        for (uint32_t t = 0; t < kI8Threads; ++t) i8_dec_load(g, tile, (uint32_t)b, t);
        for (uint32_t t = 0; t < kI8Threads; ++t) i8_dec_store<OT>(g, tile, (uint32_t)b, t);
    }
}

// bytes per element of a decoder output type (the library's alignment
// rules: four elements per vector store)
static int esize_of(int32_t out_dtype) {
    return out_dtype == BB_F16 || out_dtype == BB_BF16 ? 2 : 4;
}

extern "C" {

const char *emu_reduced_error(void) { return g_err_typed.c_str(); }

int bb_decode_bitfield_typed(const void *src, const int64_t *unit_offset,
                             int64_t nset, int32_t nthread,
                             int64_t payload_nbytes, int32_t bps,
                             int32_t nelem, int32_t complex_data,
                             int32_t codec, const float *levels_host,
                             float fill_value, int64_t sample_start,
                             int64_t nsample, int32_t out_dtype, void *out,
                             void *stream) {
    std::vector<DecLaunch> launches;
    if (!plan_decode(src, unit_offset, nset, nthread, payload_nbytes, bps,
                     nelem, complex_data, fill_value, sample_start, nsample,
                     out, launches, g_err_typed))
        return BB_ERR_ARGUMENT;
    if (out_dtype == BB_F16)
        return typed_dispatch<F16>(bps, codec, levels_host, launches);
    if (out_dtype == BB_BF16)
        return typed_dispatch<BF16>(bps, codec, levels_host, launches);
    return typed_dispatch<float>(bps, codec, levels_host, launches);
}

int bb_mark4_decode_typed(const void *src, const int64_t *unit_offset,
                          int64_t nframe, int32_t nchan, int32_t fanout,
                          int32_t ft, const float *levels_host,
                          float fill_value, int64_t sample_start,
                          int64_t nsample, int32_t out_dtype, void *out,
                          void *stream) {
    std::vector<M4Launch> l;
    if (!plan_m4_frames(false, src, unit_offset, nframe, nchan, fanout, ft,
                        levels_host, fill_value, sample_start, nsample, out,
                        nullptr, l, g_err_typed))
        return BB_ERR_ARGUMENT;
    if (out_dtype == BB_F16) typed_mark4<F16>(l);
    else if (out_dtype == BB_BF16) typed_mark4<BF16>(l);
    else typed_mark4<float>(l);
    return 0;
}

int bb_decode_int8_transposed_typed(const void *src,
                                    const int64_t *unit_offset, int64_t nunit,
                                    int64_t nrow, int64_t ncol,
                                    int32_t item_nbytes,
                                    const int64_t *col_begin,
                                    const int64_t *col_end,
                                    const int64_t *out_col0,
                                    int32_t out_dtype, void *out,
                                    void *stream) {
    if (item_nbytes != 1 && item_nbytes != 2) return BB_ERR_ARGUMENT;
    const bool fast = nrow % 2 == 0
        && (reinterpret_cast<uintptr_t>(out) % (4 * esize_of(out_dtype))) == 0;
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
    g.src = (const uint8_t *)src;
    g.unit_offset = (const long long *)unit_offset;
    g.col_begin = (const long long *)col_begin;
    g.col_end = (const long long *)col_end;
    g.out_col0 = (const long long *)out_col0;
    g.out = out; g.in = nullptr;
    if (out_dtype == BB_F16) typed_int8_t<F16>(g, nblocks, fast);
    else if (out_dtype == BB_BF16) typed_int8_t<BF16>(g, nblocks, fast);
    else typed_int8_t<float>(g, nblocks, fast);
    return 0;
}

int bb_decode_int8_timefirst_typed(const void *src,
                                   const int64_t *unit_offset, int64_t nunit,
                                   int64_t nsample, int32_t nchan,
                                   int32_t npol, int32_t item_nbytes,
                                   const int64_t *t_begin,
                                   const int64_t *t_end,
                                   const int64_t *out_t0, int32_t out_dtype,
                                   void *out, void *stream) {
    TFGeom g;
    if (tf_fill_geom(g, nunit, nsample, nchan, npol, item_nbytes,
                     (reinterpret_cast<uintptr_t>(out)
                      % (4 * esize_of(out_dtype))) == 0))
        return BB_ERR_ARGUMENT;
    g.src = (const uint8_t *)src;
    g.unit_offset = (const long long *)unit_offset;
    g.t_begin = (const long long *)t_begin;
    g.t_end = (const long long *)t_end;
    g.out_t0 = (const long long *)out_t0;
    g.out = out; g.in = nullptr;
    for (uint32_t u = 0; u < g.nunit; ++u)
        for (uint32_t i = 0; i < g.items_per_unit; ++i) {
            if (out_dtype == BB_F16) tf_decode<F16>(g, u, i);
            else if (out_dtype == BB_BF16) tf_decode<BF16>(g, u, i);
            else tf_decode<float>(g, u, i);
        }
    return 0;
}

// The host rounding the emulation stores with (bb_common.cuh): n float32
// values -> 16-bit patterns of half (brain = 0) or bfloat16 (brain = 1).
void emu_round_half(const float *in, int64_t n, int32_t brain,
                    uint16_t *out) {
    for (int64_t i = 0; i < n; ++i) {
        const uint32_t x = float_as_uint(in[i]);
        out[i] = brain ? f32_to_bf16_bits(x) : f32_to_f16_bits(x);
    }
}

}  // extern "C"
