// Generic bit-field decode/encode kernels and their C entry points.
// sm_100a only.  Streaming, HBM-bound: no tensor cores by design.
#include <string>
#include <vector>
#include "bb_runtime.cuh"
#include "bb_bitfield_plan.h"

namespace bb {

constexpr int kBlock = 256;

// Launch shape.  Measured on B200 (profiles/r1_grid_sweep.txt): for these
// write-dominated streams a plain one-shot grid in which every CTA produces a
// compact ~64 KiB tile of output beats a persistent grid-stride loop by ~18 %
// (6.4 vs 5.4 TB/s), and tiny CTAs (4 KiB) are far worse.  So every thread
// handles kUnroll items, kBlock apart, sized so a thread writes ~16 float4.
template <int BPS, int MODE>
struct Unroll {
    static constexpr int kF4PerItem =
        MODE == MODE_ROWGROUP4 ? RowSplit<BPS, 4>::kRows
        : MODE == MODE_ROWGROUP2 ? RowSplit<BPS, 2>::kRows
        : MODE == MODE_WORDRUN ? 8 / BPS
        : MODE == MODE_WORDROW4 ? 32 / BPS
        : MODE == MODE_WORDROW2 ? 16 / BPS
        : MODE == MODE_WORDROW4X2 ? 64 / BPS
        : MODE == MODE_WORDROW2X2 ? 32 / BPS
        : MODE == MODE_RUNS ? 4 : 1;
    // float4 stores per thread.  Measured (profiles/README.md, per-thread
    // work sweep): the warp-cooperative modes are 2-3 % faster with 8 than
    // with 16 (WORDRUN 6.44 -> 6.63 TB/s, above the copy rate) and slower
    // again with 4; RUN and the two-complex-thread WORDROW2 at 4/8 bit want
    // 16.  -DBB_F4_PER_THREAD=n overrides for experiments.
#ifdef BB_F4_PER_THREAD
    static constexpr int kTarget = BB_F4_PER_THREAD;
#else
    static constexpr int kTarget =
        (MODE == MODE_WORDRUN || MODE == MODE_WORDROW4
         || MODE == MODE_ROWGROUP4 || MODE == MODE_ROWGROUP2
         || (MODE == MODE_WORDROW2 && BPS <= 2)) ? 8 : 16;
#endif
    static constexpr int value = kF4PerItem >= kTarget
        ? 1 : kTarget / kF4PerItem;
};

// Encode: ROWGROUP as decode; ROWWORD sized so a warp reads ~8 KiB of rows
// per chunk and a CTA ~64 KiB; word-per-thread modes take 4 words.
template <int BPS, int MODE>
struct EncUnroll {
    static constexpr int kTpw = MODE == MODE_ROWWORD4 ? 32 / BPS : 16 / BPS;
    static constexpr int kRowF4 = (MODE == MODE_ROWGROUP4 ? 32 : 16) / BPS;
    static constexpr int value =
        (MODE == MODE_ROWGROUP4 || MODE == MODE_ROWGROUP2)
        ? (kRowF4 >= 16 ? 1 : 16 / kRowF4)
        : (MODE == MODE_ROWWORD4 || MODE == MODE_ROWWORD2)
        ? (kTpw >= 16 ? 1 : 16 / kTpw) : 4;
};

inline unsigned tile_grid(uint32_t nitems, int unroll) {
    uint64_t per_cta = (uint64_t)kBlock * unroll;
    return (unsigned)((nitems + per_cta - 1) / per_cta);
}

// The decode table lives in shared memory (see DecodeLut): built per CTA from
// the per-code levels in the kernel parameters (at most 256 floats).
template <int BPS, int CODEC, int MODE, bool SEL, typename OT>
__global__ void __launch_bounds__(kBlock)
k_decode_bitfield(const DecGeom p, const LevelTable<BPS> lv) {
    using Lut = DecodeLut<BPS>;
    constexpr int U = Unroll<BPS, MODE>::value;
    __shared__ __align__(128) float lut[CODEC == CODEC_LEVELS ? Lut::kFloats : 2];
    if (CODEC == CODEC_LEVELS && !SEL) {
        for (int i = threadIdx.x; i < Lut::kFloats; i += kBlock)
            lut[i] = Lut::value(lv.v, i);
        __syncthreads();
    }
    const uint32_t item0 = blockIdx.x * (kBlock * U) + threadIdx.x;
    if (MODE == MODE_WORDRUN) {
        // kBlock and nitems are multiples of 32, so `live` is warp uniform.
        constexpr int F = 8 / BPS;
        constexpr int B = U < 4 ? U : 4;          // chunks loaded up front
        const uint32_t lane = threadIdx.x & 31u;
#pragma unroll 1
        for (int u0 = 0; u0 < U; u0 += B) {
            uint32_t w[B];
            bool ok[B];
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const uint32_t item = item0 + (u0 + b) * kBlock;
                ok[b] = item < p.nitems && wr_load(p, item >> 5, lane, w[b]);
            }
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const uint32_t item = item0 + (u0 + b) * kBlock;
                if (item >= p.nitems) break;
                const unsigned okmask = __ballot_sync(0xffffffffu, ok[b]);
#pragma unroll
                for (int j = 0; j < F; ++j) {
                    const uint32_t src = wr_src_lane<BPS>(lane, j);
                    const uint32_t ws = __shfl_sync(0xffffffffu, w[b], src);
                    wr_emit<BPS, CODEC, OT>(p, lut, item >> 5, lane, j, ws,
                                            (okmask >> src) & 1u);
                }
            }
        }
        return;
    }
    if (MODE == MODE_WORDROW4 || MODE == MODE_WORDROW2
        || MODE == MODE_WORDROW4X2 || MODE == MODE_WORDROW2X2) {
        // The slot words of every lane go through shared memory (one vector
        // store per lane and chunk); a float4 then costs one LDS.128 / LDS.64
        // instead of G + 1 shuffles.
        constexpr int G = (MODE == MODE_WORDROW4 || MODE == MODE_WORDROW4X2)
            ? 4 : 2;
        constexpr int NG = (MODE == MODE_WORDROW4X2
                            || MODE == MODE_WORDROW2X2) ? 2 : 1;
        constexpr int W = G * NG;                 // words (slots) per row
        constexpr int TPW = (32 / BPS) / (4 / G);
        constexpr int NST = TPW * NG;             // stores per lane and chunk
        constexpr int WB = U < 2 ? U : 2;         // chunks loaded up front
        __shared__ __align__(16) uint32_t wbuf[kBlock / 32][WB][32][W];
        __shared__ uint32_t okbuf[kBlock / 32][WB][32];
        const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll 1
        for (int u0 = 0; u0 < U; u0 += WB) {
            __syncwarp();                         // previous batch consumed
#pragma unroll
            for (int b = 0; b < WB; ++b) {
                const uint32_t item = item0 + (u0 + b) * kBlock;
                uint32_t w[W];
                uint32_t ok = 0u;
#pragma unroll
                for (int g = 0; g < W; ++g) w[g] = 0u;
                if (item < p.nitems) ok = wrow_load<W>(p, item >> 5, lane, w);
#pragma unroll
                for (int g = 0; g < W; ++g) wbuf[warp][b][lane][g] = w[g];
                okbuf[warp][b][lane] = ok;
            }
            __syncwarp();
#pragma unroll
            for (int b = 0; b < WB; ++b) {
                const uint32_t item = item0 + (u0 + b) * kBlock;
                if (item >= p.nitems) break;
                // two separate loops: the interior one stays free of the
                // edge path's bounds arithmetic
                if (wrow_interior<BPS, G>(p, item >> 5)) {   // warp uniform
                    OT *chunk_out = wrow_chunk_out<BPS, G, NG, OT>(p,
                                                                   item >> 5);
#pragma unroll
                    for (int j = 0; j < NST; ++j) {
                        const uint32_t q = lane + 32u * j;
                        const uint32_t src = wrow_src_lane<BPS, G, NG>(lane,
                                                                       j);
                        const uint32_t grp = q % NG;
                        uint32_t ws[G];
#pragma unroll
                        for (int g = 0; g < G; ++g)
                            ws[g] = wbuf[warp][b][src][grp * G + g];
                        wrow_emit_fast<BPS, CODEC, G, NG>(
                            p, lut, chunk_out, q, ws,
                            (okbuf[warp][b][src] >> (grp * G))
                            & ((1u << G) - 1u));
                    }
                    continue;
                }
#pragma unroll
                for (int j = 0; j < NST; ++j) {
                    const uint32_t q = lane + 32u * j;
                    const uint32_t src = wrow_src_lane<BPS, G, NG>(lane, j);
                    const uint32_t grp = q % NG;
                    uint32_t ws[G];
#pragma unroll
                    for (int g = 0; g < G; ++g)
                        ws[g] = wbuf[warp][b][src][grp * G + g];
                    wrow_emit<BPS, CODEC, G, NG, OT>(
                        p, lut, item >> 5, lane, j, ws,
                        (okbuf[warp][b][src] >> (grp * G))
                        & ((1u << G) - 1u));
                }
            }
        }
        return;
    }
    // Batches of B items: all loads of a batch are issued before the first
    // item is decoded (memory-level parallelism).
    constexpr int B = U < 4 ? U : 4;
    if (MODE == MODE_ROWGROUP4 || MODE == MODE_ROWGROUP2) {
        constexpr int G = MODE == MODE_ROWGROUP4 ? 4 : 2;
#ifndef BB_ROW_BATCH
#define BB_ROW_BATCH 2
#endif
        constexpr int RB = U < BB_ROW_BATCH ? U : BB_ROW_BATCH;
#pragma unroll 1
        for (int u0 = 0; u0 < U; u0 += RB) {
            RowItem<G> it[RB];
#pragma unroll
            for (int b = 0; b < RB; ++b) {
                const uint32_t item = item0 + (u0 + b) * kBlock;
                it[b].live = false;
                if (item < p.nitems) rowgroup_fetch<BPS, G>(p, item, it[b]);
            }
#pragma unroll
            for (int b = 0; b < RB; ++b)
                rowgroup_emit<BPS, CODEC, G, SEL, OT>(p, lut, it[b], lv);
        }
        return;
    }
    if (MODE == MODE_RUNS) {
#pragma unroll 1
        for (int u0 = 0; u0 < U; u0 += B) {
            RunsItem it[B];
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const uint32_t item = item0 + (u0 + b) * kBlock;
                it[b].gidx = -1;
                if (item < p.nitems) runs_fetch<BPS>(p, item, it[b]);
            }
#pragma unroll
            for (int b = 0; b < B; ++b)
                runs_emit<BPS, CODEC, OT>(p, lut, it[b]);
        }
        return;
    }
    if (MODE == MODE_RUN) {
#pragma unroll 1
        for (int u0 = 0; u0 < U; u0 += B) {
            RunItem it[B];
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const uint32_t item = item0 + (u0 + b) * kBlock;
                it[b].gidx = -1;
                if (item < p.nitems) run_fetch<BPS>(p, item, it[b]);
            }
#pragma unroll
            for (int b = 0; b < B; ++b) run_emit<BPS, CODEC, OT>(p, lut, it[b]);
        }
        return;
    }
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
        const uint32_t item = item0 + u * kBlock;
        if (item >= p.nitems) break;
        dec_scalar<BPS, CODEC, OT>(p, lut, item);
    }
}

// TILE (rows of four float4, see bb_bitfield.cuh): warp-cooperative, words
// staged in shared memory, every store instruction 512 contiguous bytes.
template <int BPS, int CODEC, int G, int P, bool SEL, int U, typename OT>
__global__ void __launch_bounds__(kBlock)
k_decode_tile(const DecGeom p, const LevelTable<BPS> lv) {
    using Lut = DecodeLut<BPS>;
    using T = Tile<BPS, G, P>;
    constexpr int UB = U < 2 ? U : 2;             // chunks loaded up front
    __shared__ __align__(128) float lut[(CODEC == CODEC_LEVELS && !SEL)
                                        ? Lut::kFloats : 2];
    __shared__ __align__(16) uint32_t wbuf[kBlock / 32][UB][T::kWords];
    __shared__ uint32_t okbuf[kBlock / 32][UB][32];
    if (CODEC == CODEC_LEVELS && !SEL) {
        for (int i = threadIdx.x; i < Lut::kFloats; i += kBlock)
            lut[i] = Lut::value(lv.v, i);
        __syncthreads();
    }
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t item0 = blockIdx.x * (kBlock * U) + threadIdx.x;
#pragma unroll 1
    for (int u0 = 0; u0 < U; u0 += UB) {
        __syncwarp();                             // previous batch consumed
        bool full[UB];
#pragma unroll
        for (int b = 0; b < UB; ++b) {
            const uint32_t item = item0 + (u0 + b) * kBlock;
            uint32_t w[T::kNl];
            uint32_t ok = 0u;
#pragma unroll
            for (int i = 0; i < T::kNl; ++i) w[i] = 0u;
            if (item < p.nitems) ok = tile_load<BPS, G, P>(p, item >> 5, lane, w);
#pragma unroll
            for (int i = 0; i < T::kNl; ++i)
                wbuf[warp][b][T::kNl * lane + i] = w[i];
            full[b] = __all_sync(0xffffffffu, ok == (1u << T::kNl) - 1u);
            if (!full[b]) okbuf[warp][b][lane] = ok;
        }
        __syncwarp();
#pragma unroll
        for (int b = 0; b < UB; ++b) {
            const uint32_t item = item0 + (u0 + b) * kBlock;
            if (item >= p.nitems) break;          // warp uniform
            const uint32_t chunk = item >> 5;
            if (full[b] && tile_interior<BPS, G, P>(p, chunk)) {
                OT *chunk_out = tile_chunk_out<BPS, G, P, OT>(p, chunk);
#pragma unroll
                for (int j = 0; j < T::kStores; ++j) {
                    const uint32_t q = lane + 32u * j;
                    const uint32_t at = ((q >> 2) / T::kTpw) * T::kSlots
                        + (q & 3u) * G;
                    uint32_t ws[G];
#pragma unroll
                    for (int g = 0; g < G; ++g) ws[g] = wbuf[warp][b][at + g];
                    store4(chunk_out + 4u * q,
                           tile_decode<BPS, CODEC, G, P, SEL>(q, ws, lut, lv));
                }
                continue;
            }
#pragma unroll 1
            for (int j = 0; j < T::kStores; ++j) {
                const uint32_t q = lane + 32u * j;
                const uint32_t at = ((q >> 2) / T::kTpw) * T::kSlots
                    + (q & 3u) * G;
                uint32_t ws[G];
#pragma unroll
                for (int g = 0; g < G; ++g) ws[g] = wbuf[warp][b][at + g];
                const uint32_t okm = full[b] ? (1u << G) - 1u
                    : tile_group_ok<BPS, G, P>(okbuf[warp][b], q);
                tile_emit<BPS, CODEC, G, P, SEL, OT>(p, lut, lv, chunk, q, ws,
                                                     okm);
            }
        }
    }
}

// ROWWORD (rows of one float4 -> words through shared memory).  A kernel of
// its own so that it can carry a min-blocks hint of 4 (<= 64 registers): that
// lets ptxas keep the eight float4 loads of a lane in flight instead of
// serialising them to stay within 40 registers.
template <typename S, int BPS, int QUANT, int G>
__global__ void __launch_bounds__(kBlock, 4)
k_encode_rowword(const EncGeom p, const QuantConsts<arith_t<S>> c) {
    constexpr int MODE = G == 4 ? MODE_ROWWORD4 : MODE_ROWWORD2;
    constexpr int U = EncUnroll<BPS, MODE>::value;
    constexpr int TPW = (32 / BPS) / (4 / G);
    __shared__ uint32_t cbuf[kBlock / 32][32 * TPW];
    // kBlock and nitems are multiples of 32: chunks are warp uniform.
    const uint32_t item0 = blockIdx.x * (kBlock * U) + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
        const uint32_t item = item0 + u * kBlock;
        if (item >= p.nitems) break;
        rw_stage<S, BPS, QUANT, G>(p, c, item >> 5, lane, cbuf[warp]);
        __syncwarp();
        rw_emit<BPS, G>(p, item >> 5, lane, cbuf[warp]);
        __syncwarp();                             // before the buffer is reused
    }
}

template <typename S, int BPS, int QUANT, int MODE>
__global__ void __launch_bounds__(kBlock)
k_encode_bitfield(const EncGeom p, const QuantConsts<arith_t<S>> c) {
    using T = arith_t<S>;
    constexpr int U = EncUnroll<BPS, MODE>::value;
    const uint32_t item0 = blockIdx.x * (kBlock * U) + threadIdx.x;
    if (MODE == MODE_RUNQ) {
        // four words per item: two items' (eight) loads in flight (float
        // arithmetic; one for float64)
        constexpr int B = sizeof(T) == 4 ? 2 : 1;
#pragma unroll 1
        for (int u0 = 0; u0 < U; u0 += B) {
            EncQuadItem<T> it[B];
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const uint32_t item = item0 + (u0 + b) * kBlock;
                it[b].dst = nullptr;
                if (item < p.nitems) enc_quad_fetch<S>(p, item, it[b]);
            }
#pragma unroll
            for (int b = 0; b < B; ++b) enc_quad_emit<T, QUANT>(c, it[b]);
        }
        return;
    }
    if (MODE == MODE_RUN && BPS >= 4) {
        // few float4 per word: keep the loads of several words in flight
        constexpr int B = BPS == 8 ? 4 : 2;
#pragma unroll 1
        for (int u0 = 0; u0 < U; u0 += B) {
            EncWordItem<T, BPS> it[B];
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const uint32_t item = item0 + (u0 + b) * kBlock;
                it[b].dst = nullptr;
                if (item < p.nitems) enc_word_fetch<S, BPS>(p, item, it[b]);
            }
#pragma unroll
            for (int b = 0; b < B; ++b)
                enc_word_emit<T, BPS, QUANT>(c, it[b]);
        }
        return;
    }
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
        const uint32_t item = item0 + u * kBlock;
        if (item >= p.nitems) break;
        if (MODE == MODE_ROWGROUP4) enc_rowgroup<S, BPS, QUANT, 4>(p, c, item);
        else if (MODE == MODE_ROWGROUP2) enc_rowgroup<S, BPS, QUANT, 2>(p, c, item);
        else if (MODE == MODE_RUN) enc_word<S, BPS, QUANT, true>(p, c, item);
        else enc_word<S, BPS, QUANT, false>(p, c, item);
    }
}

// The 2-bit level-table variants under evaluation (register select, TILE).
// Returns false if the launch is not one of them.
template <int BPS, int CODEC, int G, int P, bool SEL, typename OT>
static void launch_tile(const DecLaunch &l, const LevelTable<BPS> &lv,
                        cudaStream_t stream) {
    if (l.tile_u >= 2)
        k_decode_tile<BPS, CODEC, G, P, SEL, 2, OT>
            <<<tile_grid(l.g.nitems, 2), kBlock, 0, stream>>>(l.g, lv);
    else
        k_decode_tile<BPS, CODEC, G, P, SEL, 1, OT>
            <<<tile_grid(l.g.nitems, 1), kBlock, 0, stream>>>(l.g, lv);
}

template <int BPS, int CODEC, typename OT>
static bool launch_c2(const DecLaunch &l, const LevelTable<BPS> &lv,
                      cudaStream_t stream) {
    const uint32_t n = l.g.nitems;
    if (l.mode == MODE_ROWGROUP4 && l.sel) {
        k_decode_bitfield<BPS, CODEC, MODE_ROWGROUP4, true, OT>
            <<<tile_grid(n, Unroll<BPS, MODE_ROWGROUP4>::value), kBlock, 0,
               stream>>>(l.g, lv);
        return true;
    }
    if (l.mode == MODE_ROWGROUP2 && l.sel) {
        k_decode_bitfield<BPS, CODEC, MODE_ROWGROUP2, true, OT>
            <<<tile_grid(n, Unroll<BPS, MODE_ROWGROUP2>::value), kBlock, 0,
               stream>>>(l.g, lv);
        return true;
    }
    if (l.mode == MODE_TILE4) {
        if (l.tile_p == 8 && l.sel) launch_tile<BPS, CODEC, 4, 8, true, OT>(l, lv, stream);
        else if (l.tile_p == 8) launch_tile<BPS, CODEC, 4, 8, false, OT>(l, lv, stream);
        else if (l.sel) launch_tile<BPS, CODEC, 4, 4, true, OT>(l, lv, stream);
        else launch_tile<BPS, CODEC, 4, 4, false, OT>(l, lv, stream);
        return true;
    }
    if (l.mode == MODE_TILE2) {
        if (l.tile_p == 8 && l.sel) launch_tile<BPS, CODEC, 2, 8, true, OT>(l, lv, stream);
        else if (l.tile_p == 8) launch_tile<BPS, CODEC, 2, 8, false, OT>(l, lv, stream);
        else if (l.sel) launch_tile<BPS, CODEC, 2, 4, true, OT>(l, lv, stream);
        else launch_tile<BPS, CODEC, 2, 4, false, OT>(l, lv, stream);
        return true;
    }
    return false;
}

template <int BPS, int CODEC, typename OT>
static int launch_decode(const std::vector<DecLaunch> &launches,
                         const float *levels_host, cudaStream_t stream) {
    LevelTable<BPS> lv;
    for (int i = 0; i < (1 << BPS); ++i)
        lv.v[i] = (CODEC == CODEC_LEVELS && levels_host) ? levels_host[i] : 0.f;
    for (const DecLaunch &l : launches) {
        const uint32_t n = l.g.nitems;
        if constexpr (BPS == 2 && CODEC == CODEC_LEVELS) {
            if (launch_c2<BPS, CODEC, OT>(l, lv, stream)) {
                BB_CHECK_LAUNCH("bb_decode_bitfield launch");
                continue;
            }
        }
        switch (l.mode) {
        case MODE_ROWGROUP4:
            k_decode_bitfield<BPS, CODEC, MODE_ROWGROUP4, false, OT>
                <<<tile_grid(n, Unroll<BPS, MODE_ROWGROUP4>::value), kBlock, 0,
                   stream>>>(l.g, lv);
            break;
        case MODE_ROWGROUP2:
            k_decode_bitfield<BPS, CODEC, MODE_ROWGROUP2, false, OT>
                <<<tile_grid(n, Unroll<BPS, MODE_ROWGROUP2>::value), kBlock, 0,
                   stream>>>(l.g, lv);
            break;
        case MODE_RUN:
            k_decode_bitfield<BPS, CODEC, MODE_RUN, false, OT>
                <<<tile_grid(n, Unroll<BPS, MODE_RUN>::value), kBlock, 0,
                   stream>>>(l.g, lv);
            break;
        case MODE_RUNS:
            k_decode_bitfield<BPS, CODEC, MODE_RUNS, false, OT>
                <<<tile_grid(n, Unroll<BPS, MODE_RUNS>::value), kBlock, 0,
                   stream>>>(l.g, lv);
            break;
        case MODE_WORDRUN:
            k_decode_bitfield<BPS, CODEC, MODE_WORDRUN, false, OT>
                <<<tile_grid(n, Unroll<BPS, MODE_WORDRUN>::value), kBlock, 0,
                   stream>>>(l.g, lv);
            break;
        case MODE_WORDROW4:
            k_decode_bitfield<BPS, CODEC, MODE_WORDROW4, false, OT>
                <<<tile_grid(n, Unroll<BPS, MODE_WORDROW4>::value), kBlock, 0,
                   stream>>>(l.g, lv);
            break;
        case MODE_WORDROW2:
            k_decode_bitfield<BPS, CODEC, MODE_WORDROW2, false, OT>
                <<<tile_grid(n, Unroll<BPS, MODE_WORDROW2>::value), kBlock, 0,
                   stream>>>(l.g, lv);
            break;
        case MODE_WORDROW4X2:
            k_decode_bitfield<BPS, CODEC, MODE_WORDROW4X2, false, OT>
                <<<tile_grid(n, Unroll<BPS, MODE_WORDROW4X2>::value), kBlock,
                   0, stream>>>(l.g, lv);
            break;
        case MODE_WORDROW2X2:
            k_decode_bitfield<BPS, CODEC, MODE_WORDROW2X2, false, OT>
                <<<tile_grid(n, Unroll<BPS, MODE_WORDROW2X2>::value), kBlock,
                   0, stream>>>(l.g, lv);
            break;
        default:
            k_decode_bitfield<BPS, CODEC, MODE_SCALAR, false, OT>
                <<<tile_grid(n, Unroll<BPS, MODE_SCALAR>::value), kBlock, 0,
                   stream>>>(l.g, lv);
        }
        BB_CHECK_LAUNCH("bb_decode_bitfield launch");
    }
    return BB_OK;
}

template <typename S, int BPS, int QUANT>
static int launch_encode(const std::vector<EncLaunch> &launches,
                         cudaStream_t stream) {
    using T = arith_t<S>;
    static const QuantConsts<T> consts = make_quant_consts<T>();
    for (const EncLaunch &l : launches) {
        const uint32_t n = l.g.nitems;
        switch (l.mode) {
        case MODE_ROWGROUP4:
            k_encode_bitfield<S, BPS, QUANT, MODE_ROWGROUP4>
                <<<tile_grid(n, EncUnroll<BPS, MODE_ROWGROUP4>::value), kBlock,
                   0, stream>>>(l.g, consts);
            break;
        case MODE_ROWGROUP2:
            k_encode_bitfield<S, BPS, QUANT, MODE_ROWGROUP2>
                <<<tile_grid(n, EncUnroll<BPS, MODE_ROWGROUP2>::value), kBlock,
                   0, stream>>>(l.g, consts);
            break;
        case MODE_ROWWORD4:
            k_encode_rowword<S, BPS, QUANT, 4>
                <<<tile_grid(n, EncUnroll<BPS, MODE_ROWWORD4>::value), kBlock,
                   0, stream>>>(l.g, consts);
            break;
        case MODE_ROWWORD2:
            k_encode_rowword<S, BPS, QUANT, 2>
                <<<tile_grid(n, EncUnroll<BPS, MODE_ROWWORD2>::value), kBlock,
                   0, stream>>>(l.g, consts);
            break;
        case MODE_RUN:
            k_encode_bitfield<S, BPS, QUANT, MODE_RUN>
                <<<tile_grid(n, 4), kBlock, 0, stream>>>(l.g, consts);
            break;
        case MODE_RUNQ:
            if constexpr (BPS == 8)
                k_encode_bitfield<S, 8, QUANT, MODE_RUNQ>
                    <<<tile_grid(n, 4), kBlock, 0, stream>>>(l.g, consts);
            break;
        default:
            k_encode_bitfield<S, BPS, QUANT, MODE_SCALAR>
                <<<tile_grid(n, 4), kBlock, 0, stream>>>(l.g, consts);
        }
        BB_CHECK_LAUNCH("bb_encode_bitfield launch");
    }
    return BB_OK;
}

template <typename S>
static int dispatch_encode(int bps, int quantiser,
                           const std::vector<EncLaunch> &l, cudaStream_t s) {
    if (quantiser == BB_QUANT_OFFSET_BINARY) {
        switch (bps) {
        case 1: return launch_encode<S, 1, QUANT_OFFSET>(l, s);
        case 2: return launch_encode<S, 2, QUANT_OFFSET>(l, s);
        case 4: return launch_encode<S, 4, QUANT_OFFSET>(l, s);
        case 8: return launch_encode<S, 8, QUANT_OFFSET>(l, s);
        }
    } else if (quantiser == BB_QUANT_MARK5B) {
        switch (bps) {
        case 1: return launch_encode<S, 1, QUANT_MARK5B>(l, s);
        case 2: return launch_encode<S, 2, QUANT_MARK5B>(l, s);
        }
    } else if (quantiser == BB_QUANT_SINT) {
        switch (bps) {
        case 4: return launch_encode<S, 4, QUANT_SINT>(l, s);
        case 8: return launch_encode<S, 8, QUANT_SINT>(l, s);
        }
    }
    return set_error(BB_ERR_UNSUPPORTED,
                     "cannot encode data with %d bits (quantiser %d)", bps,
                     quantiser);
}

template <typename OT>
static int dispatch_decode(int bps, int codec, const float *levels_host,
                           const std::vector<DecLaunch> &l, cudaStream_t s) {
    if (codec == BB_CODEC_LEVELS) {
        switch (bps) {
        case 1: return launch_decode<1, CODEC_LEVELS, OT>(l, levels_host, s);
        case 2: return launch_decode<2, CODEC_LEVELS, OT>(l, levels_host, s);
        case 4: return launch_decode<4, CODEC_LEVELS, OT>(l, levels_host, s);
        case 8:
            if (affine8_matches(levels_host))       // the standard 8-bit table
                return launch_decode<8, CODEC_AFFINE8, OT>(l, nullptr, s);
            return launch_decode<8, CODEC_LEVELS, OT>(l, levels_host, s);
        }
    } else if (codec == BB_CODEC_SINT) {
        switch (bps) {
        case 4: return launch_decode<4, CODEC_SINT, OT>(l, nullptr, s);
        case 8: return launch_decode<8, CODEC_SINT, OT>(l, nullptr, s);
        }
    }
    return set_error(BB_ERR_UNSUPPORTED, "no decoder for bps=%d codec=%d", bps,
                     codec);
}

}  // namespace bb

using namespace bb;

extern "C" int bb_decode_bitfield_typed(
    const void *src, const int64_t *unit_offset, int64_t nset, int32_t nthread,
    int64_t payload_nbytes, int32_t bps, int32_t nelem, int32_t complex_data,
    int32_t codec, const float *levels_host, float fill_value,
    int64_t sample_start, int64_t nsample, int32_t out_dtype, void *out,
    void *stream) {
    if (!src || !unit_offset || !out)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    const int esize = out_elem_nbytes(out_dtype);
    if (esize == 0)
        return set_error(BB_ERR_ARGUMENT,
                         "out_dtype must be BB_F32, BB_F16 or BB_BF16");
    const int out_align = 4 * esize;             // one float4-equivalent
    if (!aligned(out, out_align) || !aligned(src, 4))
        return set_error(BB_ERR_ALIGNMENT,
                         "out must be %d-byte and src 4-byte aligned",
                         out_align);
    if (codec == BB_CODEC_LEVELS && !levels_host)
        return set_error(BB_ERR_ARGUMENT, "levels_host required");
    std::vector<DecLaunch> launches;
    std::string err;
    if (!plan_decode(src, unit_offset, nset, nthread, payload_nbytes, bps,
                     nelem, complex_data, fill_value, sample_start, nsample,
                     out, launches, err))
        return set_error(BB_ERR_ARGUMENT, "%s", err.c_str());
    cudaStream_t s = as_stream(stream);
    if (out_dtype == BB_F16)
        return dispatch_decode<F16>(bps, codec, levels_host, launches, s);
    if (out_dtype == BB_BF16)
        return dispatch_decode<BF16>(bps, codec, levels_host, launches, s);
    return dispatch_decode<float>(bps, codec, levels_host, launches, s);
}

extern "C" int bb_decode_bitfield(
    const void *src, const int64_t *unit_offset, int64_t nset, int32_t nthread,
    int64_t payload_nbytes, int32_t bps, int32_t nelem, int32_t complex_data,
    int32_t codec, const float *levels_host, float fill_value,
    int64_t sample_start, int64_t nsample, float *out, void *stream) {
    return bb_decode_bitfield_typed(src, unit_offset, nset, nthread,
                                    payload_nbytes, bps, nelem, complex_data,
                                    codec, levels_host, fill_value,
                                    sample_start, nsample, BB_F32, out,
                                    stream);
}

extern "C" int bb_encode_bitfield_typed(
    const void *in, int32_t in_dtype, void *dst, const int64_t *unit_offset,
    int64_t nset, int32_t nthread, int64_t payload_nbytes, int32_t bps,
    int32_t nelem, int32_t quantiser, void *stream) {
    if (!in || !dst || !unit_offset)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    const int in_align = in_vec_align(in_dtype);
    if (in_align == 0)
        return set_error(BB_ERR_ARGUMENT,
                         "in_dtype must be BB_F32, BB_F64, BB_F16 or BB_BF16");
    if (!aligned(in, in_align) || !aligned(dst, 4))
        return set_error(BB_ERR_ALIGNMENT,
                         "in must be %d-byte and dst 4-byte aligned",
                         in_align);
    std::vector<EncLaunch> launches;
    std::string err;
    if (!plan_encode(in, dst, unit_offset, nset, nthread, payload_nbytes, bps,
                     nelem, launches, err))
        return set_error(BB_ERR_ARGUMENT, "%s", err.c_str());
    cudaStream_t s = as_stream(stream);
    if (in_dtype == BB_F32) return dispatch_encode<float>(bps, quantiser, launches, s);
    if (in_dtype == BB_F64) return dispatch_encode<double>(bps, quantiser, launches, s);
    if (in_dtype == BB_F16) return dispatch_encode<F16>(bps, quantiser, launches, s);
    return dispatch_encode<BF16>(bps, quantiser, launches, s);
}

extern "C" int bb_encode_bitfield(
    const void *in, int32_t in_dtype, void *dst, const int64_t *unit_offset,
    int64_t nset, int32_t nthread, int64_t payload_nbytes, int32_t bps,
    int32_t nelem, int32_t quantiser, void *stream) {
    if (in_dtype != BB_F32 && in_dtype != BB_F64)
        return set_error(BB_ERR_ARGUMENT, "in_dtype must be BB_F32 or BB_F64");
    return bb_encode_bitfield_typed(in, in_dtype, dst, unit_offset, nset,
                                    nthread, payload_nbytes, bps, nelem,
                                    quantiser, stream);
}
