// CPU emulation of the bit-field kernels — TEST INFRASTRUCTURE ONLY.
//
// Compiles the very same per-thread bodies and launch planning that the CUDA
// library uses (baseband_b200/csrc/bb_bitfield.cuh, bb_bitfield_plan.h) with
// g++ and runs every "thread" in a loop, so the index arithmetic, the fast /
// edge paths and the quantisers can be checked against the oracle on a box
// without a GPU.  Never loaded by baseband_b200.
#include <cstring>
#include <string>
#include <vector>
#include "../../baseband_b200/csrc/bb_bitfield_plan.h"
#include "../../include/baseband_b200.h"

using namespace bb;

static std::string g_err;

// warp-cooperative WORDROW modes: the shared-memory word buffer is an array
template <int BPS, int CODEC, int G, int NG>
static void run_wordrow(const DecGeom &g, const float *lut) {
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
                        g, lut, wrow_chunk_out<BPS, G, NG>(g, chunk), q,
                        &w[src][grp * G], okg);
                else
                    wrow_emit<BPS, CODEC, G, NG>(g, lut, chunk, lane, j,
                                                 &w[src][grp * G], okg);
            }
    }
}

// warp-cooperative TILE modes
template <int BPS, int CODEC, int G, int P, bool SEL>
static void run_tile(const DecGeom &g, const float *lut, const float *levels) {
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
                *reinterpret_cast<F4 *>(tile_chunk_out<BPS, G, P>(g, chunk)
                                        + 4u * q) =
                    tile_decode<BPS, CODEC, G, P, SEL>(q, &wbuf[at], lut, lv);
            else
                tile_emit<BPS, CODEC, G, P, SEL>(
                    g, lut, lv, chunk, q, &wbuf[at],
                    full ? (1u << G) - 1u : tile_group_ok<BPS, G, P>(oks, q));
        }
    }
}

template <int BPS, int CODEC>
static void run_decode(const std::vector<DecLaunch> &launches,
                       const float *levels) {
    using Lut = DecodeLut<BPS>;
    alignas(16) float lut[Lut::kFloats];
    if (CODEC == CODEC_LEVELS)
        for (int i = 0; i < Lut::kFloats; ++i) lut[i] = Lut::value(levels, i);
    for (const DecLaunch &l : launches) {
        if (l.mode == MODE_WORDRUN) {
            // warp-cooperative mode: emulate the shuffle with a 32-word array
            constexpr int F = 8 / BPS;
            for (uint32_t chunk = 0; chunk < l.g.nitems / 32; ++chunk) {
                uint32_t w[32];
                bool ok[32];
                for (uint32_t lane = 0; lane < 32; ++lane)
                    ok[lane] = wr_load(l.g, chunk, lane, w[lane]);
                for (uint32_t lane = 0; lane < 32; ++lane)
                    for (int j = 0; j < F; ++j) {
                        uint32_t src = wr_src_lane<BPS>(lane, j);
                        wr_emit<BPS, CODEC>(l.g, lut, chunk, lane, j, w[src],
                                            ok[src]);
                    }
            }
            continue;
        }
        if (is_tile(l.mode)) {
            if constexpr (BPS == 2 && CODEC == CODEC_LEVELS) {
                const bool g4 = l.mode == MODE_TILE4;
                if (g4 && l.tile_p == 8 && l.sel) run_tile<BPS, CODEC, 4, 8, true>(l.g, lut, levels);
                else if (g4 && l.tile_p == 8) run_tile<BPS, CODEC, 4, 8, false>(l.g, lut, levels);
                else if (g4 && l.sel) run_tile<BPS, CODEC, 4, 4, true>(l.g, lut, levels);
                else if (g4) run_tile<BPS, CODEC, 4, 4, false>(l.g, lut, levels);
                else if (l.tile_p == 8 && l.sel) run_tile<BPS, CODEC, 2, 8, true>(l.g, lut, levels);
                else if (l.tile_p == 8) run_tile<BPS, CODEC, 2, 8, false>(l.g, lut, levels);
                else if (l.sel) run_tile<BPS, CODEC, 2, 4, true>(l.g, lut, levels);
                else run_tile<BPS, CODEC, 2, 4, false>(l.g, lut, levels);
            }
            continue;
        }
        if (is_wordrow(l.mode)) {
            if (l.mode == MODE_WORDROW4) run_wordrow<BPS, CODEC, 4, 1>(l.g, lut);
            else if (l.mode == MODE_WORDROW2) run_wordrow<BPS, CODEC, 2, 1>(l.g, lut);
            else if (l.mode == MODE_WORDROW4X2) run_wordrow<BPS, CODEC, 4, 2>(l.g, lut);
            else run_wordrow<BPS, CODEC, 2, 2>(l.g, lut);
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
                        rowgroup_emit<BPS, CODEC, 4, true>(l.g, lut, it, lv);
                    } else {
                        RowItem<2> it;
                        rowgroup_fetch<BPS, 2>(l.g, item, it);
                        rowgroup_emit<BPS, CODEC, 2, true>(l.g, lut, it, lv);
                    }
                }
                continue;
            }
            if (l.mode == MODE_ROWGROUP4) dec_rowgroup<BPS, CODEC, 4>(l.g, lut, item);
            else if (l.mode == MODE_ROWGROUP2) dec_rowgroup<BPS, CODEC, 2>(l.g, lut, item);
            else if (l.mode == MODE_RUN) dec_run<BPS, CODEC>(l.g, lut, item);
            else if (l.mode == MODE_RUNS) dec_runs<BPS, CODEC>(l.g, lut, item);
            else dec_scalar<BPS, CODEC>(l.g, lut, item);
        }
    }
}

template <typename T, int BPS, int QUANT>
static void run_encode(const std::vector<EncLaunch> &launches) {
    const QuantConsts<T> c = make_quant_consts<T>();
    for (const EncLaunch &l : launches) {
        if (l.mode == MODE_ROWWORD4 || l.mode == MODE_ROWWORD2) {
            // warp-cooperative mode: the staging buffer is the shared memory
            std::vector<uint32_t> buf(32 * 32);
            for (uint32_t chunk = 0; chunk < l.g.nitems / 32; ++chunk) {
                for (uint32_t lane = 0; lane < 32; ++lane) {
                    if (l.mode == MODE_ROWWORD4)
                        rw_stage<T, BPS, QUANT, 4>(l.g, c, chunk, lane, buf.data());
                    else
                        rw_stage<T, BPS, QUANT, 2>(l.g, c, chunk, lane, buf.data());
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
            if (l.mode == MODE_ROWGROUP4) enc_rowgroup<T, BPS, QUANT, 4>(l.g, c, item);
            else if (l.mode == MODE_ROWGROUP2) enc_rowgroup<T, BPS, QUANT, 2>(l.g, c, item);
            else if (l.mode == MODE_RUN) enc_word<T, BPS, QUANT, true>(l.g, c, item);
            else if (l.mode == MODE_RUNQ) {
                EncQuadItem<T> it;
                enc_quad_fetch<T>(l.g, item, it);
                enc_quad_emit<T, QUANT>(c, it);
            } else enc_word<T, BPS, QUANT, false>(l.g, c, item);
        }
    }
}

template <typename T>
static int enc_dispatch(int bps, int q, const std::vector<EncLaunch> &l) {
    if (q == BB_QUANT_OFFSET_BINARY) {
        if (bps == 1) return run_encode<T, 1, QUANT_OFFSET>(l), 0;
        if (bps == 2) return run_encode<T, 2, QUANT_OFFSET>(l), 0;
        if (bps == 4) return run_encode<T, 4, QUANT_OFFSET>(l), 0;
        if (bps == 8) return run_encode<T, 8, QUANT_OFFSET>(l), 0;
    } else if (q == BB_QUANT_MARK5B) {
        if (bps == 1) return run_encode<T, 1, QUANT_MARK5B>(l), 0;
        if (bps == 2) return run_encode<T, 2, QUANT_MARK5B>(l), 0;
    } else if (q == BB_QUANT_SINT) {
        if (bps == 4) return run_encode<T, 4, QUANT_SINT>(l), 0;
        if (bps == 8) return run_encode<T, 8, QUANT_SINT>(l), 0;
    }
    return BB_ERR_UNSUPPORTED;
}

extern "C" {

const char *bb_last_error(void) { return g_err.c_str(); }

// What the real planner makes of a call, without running it (no pointer is
// dereferenced by the planner, so the data pointers are null).  info[0] =
// mode of the first launch, info[1] = its `sel`, info[2] = the number of
// launches, info[3] = the frame sets of the first launch, info[4] = the
// items of the last launch.  Returns 0, or BB_ERR_ARGUMENT when the planner
// refuses the call.
int emu_plan_decode(int64_t nset, int32_t nthread, int64_t payload_nbytes,
                    int32_t bps, int32_t nelem, int32_t complex_data,
                    int64_t sample_start, int64_t nsample, int64_t *info) {
    std::vector<DecLaunch> launches;
    if (!plan_decode(nullptr, nullptr, nset, nthread, payload_nbytes, bps,
                     nelem, complex_data, 0.f, sample_start, nsample, nullptr,
                     launches, g_err))
        return BB_ERR_ARGUMENT;
    info[0] = launches.empty() ? -1 : launches[0].mode;
    info[1] = launches.empty() ? 0 : launches[0].sel;
    info[2] = (int64_t)launches.size();
    info[3] = launches.empty() ? 0 : launches[0].g.nset;
    info[4] = launches.empty() ? 0 : launches.back().g.nitems;
    return 0;
}

int emu_plan_encode(int64_t nset, int32_t nthread, int64_t payload_nbytes,
                    int32_t bps, int32_t nelem, int64_t *info) {
    std::vector<EncLaunch> launches;
    if (!plan_encode(nullptr, nullptr, nullptr, nset, nthread, payload_nbytes,
                     bps, nelem, launches, g_err))
        return BB_ERR_ARGUMENT;
    info[0] = launches.empty() ? -1 : launches[0].mode;
    info[1] = 0;
    info[2] = (int64_t)launches.size();
    info[3] = launches.empty() ? 0 : launches[0].g.nset;
    info[4] = launches.empty() ? 0 : launches.back().g.nitems;
    return 0;
}

int bb_decode_bitfield(const void *src, const int64_t *unit_offset,
                       int64_t nset, int32_t nthread, int64_t payload_nbytes,
                       int32_t bps, int32_t nelem, int32_t complex_data,
                       int32_t codec, const float *levels_host,
                       float fill_value, int64_t sample_start,
                       int64_t nsample, float *out, void *stream) {
    std::vector<DecLaunch> launches;
    if (!plan_decode(src, unit_offset, nset, nthread, payload_nbytes, bps,
                     nelem, complex_data, fill_value, sample_start, nsample,
                     out, launches, g_err))
        return BB_ERR_ARGUMENT;
    if (codec == BB_CODEC_LEVELS) {
        if (bps == 1) return run_decode<1, CODEC_LEVELS>(launches, levels_host), 0;
        if (bps == 2) return run_decode<2, CODEC_LEVELS>(launches, levels_host), 0;
        if (bps == 4) return run_decode<4, CODEC_LEVELS>(launches, levels_host), 0;
        if (bps == 8 && affine8_matches(levels_host))
            return run_decode<8, CODEC_AFFINE8>(launches, nullptr), 0;
        if (bps == 8) return run_decode<8, CODEC_LEVELS>(launches, levels_host), 0;
    } else {
        if (bps == 4) return run_decode<4, CODEC_SINT>(launches, nullptr), 0;
        if (bps == 8) return run_decode<8, CODEC_SINT>(launches, nullptr), 0;
    }
    return BB_ERR_UNSUPPORTED;
}

int bb_encode_bitfield(const void *in, int32_t in_dtype, void *dst,
                       const int64_t *unit_offset, int64_t nset,
                       int32_t nthread, int64_t payload_nbytes, int32_t bps,
                       int32_t nelem, int32_t quantiser, void *stream) {
    std::vector<EncLaunch> launches;
    if (!plan_encode(in, dst, unit_offset, nset, nthread, payload_nbytes, bps,
                     nelem, launches, g_err))
        return BB_ERR_ARGUMENT;
    return in_dtype == BB_F32 ? enc_dispatch<float>(bps, quantiser, launches)
                              : enc_dispatch<double>(bps, quantiser, launches);
}

}  // extern "C"

// Folded-threshold 2-bit quantiser == literal clip/add/floor_divide chain for
// every value in a neighbourhood of each threshold (and specials).
extern "C" long long emu_quant2_check(int is_double, int nulp) {
    long long bad = 0;
    if (is_double) {
        const QuantConsts<double> c = make_quant_consts<double>();
        const double marks[] = {c.x1, c.x2, c.x3, c.clip_lo, c.clip_hi, 0.0,
                                -0.0, 1e300, -1e300, INFINITY, -INFINITY, NAN};
        for (double m : marks) {
            double up = m, dn = m;
            for (int i = 0; i <= nulp; ++i) {
                bad += quant2_offset(up, c) != quant2_offset_chain(up, c);
                bad += quant2_offset(dn, c) != quant2_offset_chain(dn, c);
                up = nextafter(up, INFINITY);
                dn = nextafter(dn, -INFINITY);
            }
        }
    } else {
        const QuantConsts<float> c = make_quant_consts<float>();
        // every 1021st float of either sign, and +-nulp ulp around each
        // threshold and clip bound
        for (uint32_t bits = 0; bits < 0x7f800000u; bits += 1021u) {
            float v;
            std::memcpy(&v, &bits, 4);
            bad += quant2_offset(v, c) != quant2_offset_chain(v, c);
            bad += quant2_offset(-v, c) != quant2_offset_chain(-v, c);
        }
        const float marks[] = {c.x1, c.x2, c.x3, c.clip_lo, c.clip_hi, 0.f};
        for (float m : marks) {
            float up = m, dn = m;
            for (int i = 0; i <= nulp; ++i) {
                bad += quant2_offset(up, c) != quant2_offset_chain(up, c);
                bad += quant2_offset(dn, c) != quant2_offset_chain(dn, c);
                up = nextafterf(up, INFINITY);
                dn = nextafterf(dn, -INFINITY);
            }
        }
        const float sp[] = {1e30f, -1e30f, INFINITY, -INFINITY, NAN};
        for (float v : sp)
            bad += quant2_offset(v, c) != quant2_offset_chain(v, c);
    }
    return bad;
}

// Number of 8-bit codes for which the table-free decode differs (bitwise)
// from the level table given.
extern "C" int emu_affine8_mismatches(const float *levels) {
    int bad = 0;
    for (uint32_t code = 0; code < 256; ++code) {
        const float v = affine8(code << 16, 2);
        bad += __builtin_memcmp(&v, &levels[code], 4) != 0;
    }
    return bad + (affine8_matches(levels) ? 0 : 1000);
}
