// Generic LSB-first bit-field codec: per-thread bodies.
//
// Logical layout (see include/baseband_b200.h, bb_decode_bitfield):
//   unit (set, slot): nword 32-bit words = codes of BPS bits, LSB first, in
//                     order [time][E]   (E = nelem)
//   out:              [row][slot][E] float32 (or F16 / BF16: the emit steps
//                     are templated on the output type OT; a "float4" below
//                     is then four 16-bit values, 8 bytes),
//                     row = set*spf + t - sample_start
//
// Three work decompositions, chosen by the launcher:
//   ROWGROUP<G>  E*G == 4, nthread % G == 0.  A thread takes word k of G
//                neighbouring slots and writes, for each time in that word, one
//                float4 covering the G slots.  Lanes are ordered (group
//                fastest, then word) so every warp store covers whole rows.
//                This is the VDIF multi-thread single-channel path (C1, C2).
//   WORDRUN      nthread == 1 (Mark 5B, DADA, GSB, single-thread VDIF).  The
//                output is then one flat run of codes.  A warp takes 32
//                consecutive payload words with ONE coalesced 128-byte load,
//                and redistributes them with warp shuffles so that every
//                store instruction again covers 512 contiguous bytes (lane L
//                stores float4 L + 32 j of the warp's chunk).  Several chunks
//                are loaded before the first is decoded (memory-level
//                parallelism; the RUN mode it replaces was latency bound).
//   WORDROW<G>   nthread * E == 4: as WORDRUN over the G slots of a row.
//   RUN          nthread > 1 and E a power of two >= 4.  Output-centric: a
//                thread owns one float4 of the output (4 consecutive codes of
//                one unit), so a warp store is 512 contiguous bytes.
//   SCALAR       anything else: one output element per thread.
#pragma once
#include "bb_common.cuh"
#include "bb_quant.cuh"

namespace bb {

// CODEC_AFFINE8 is internal: the launcher substitutes it for CODEC_LEVELS when
// the 256 levels it was given are exactly those `affine8` computes.
enum { CODEC_LEVELS = 0, CODEC_SINT = 1, CODEC_AFFINE8 = 2 };

template <int BPS>
struct LevelTable { float v[1 << BPS]; };

// Decode look-up table as the kernels use it (shared memory on the device).
// For 1 and 2 bit the table is indexed by TWO adjacent codes and yields both
// values at once: 2 bit -> 16 entries x 8 B = 128 B, one entry per pair of
// banks, so a warp-wide LDS.64 never has a bank conflict; 1 bit -> 4 entries.
// 4 and 8 bit are indexed by one code (16 entries: conflict free).
template <int BPS>
struct DecodeLut {
    static constexpr int kPair = BPS <= 2;
    static constexpr int kEntries = kPair ? (1 << (2 * BPS)) : (1 << BPS);
    static constexpr int kFloats = kPair ? 2 * kEntries : kEntries;
    // entry i of the table built from per-code levels
    static BB_HD float value(const float *levels, int i) {
        if (kPair) {
            int entry = i >> 1, which = i & 1;
            int code = which ? (entry >> BPS) : (entry & ((1 << BPS) - 1));
            return levels[code];
        }
        return levels[i];
    }
};

// ------------------------------------------------------------------ decode
struct DecGeom {
    const uint8_t *src;
    const long long *unit_offset;   // [nset * nthread] for this launch
    void *out;                      // row 0 of the whole call (float32,
                                    // F16 or BF16 elements)
    long long row_base;             // row of (set 0, t 0) of this launch
    long long nsample;              // valid rows are [0, nsample)
    uint32_t nset, nthread, nelem, nword;
    uint32_t tpw;                   // times per word (ROWGROUP)
    uint32_t spf;                   // samples (times) per unit
    uint32_t nitems;
    uint32_t nwords_total;          // WORDRUN: nset * nword
    uint32_t ngroup;                // nthread / G
    int32_t log2_nelem;             // RUN with nthread > 1
    uint32_t complex_fill;
    uint32_t debug;                 // knock-out experiments (BB_TUNE_KNOCK)
    float fill;
    FastDiv div_nword, div_ngroup, div_rowlen, div_spf, div_nelem, div_unitlen;
    FastDiv div_f4row;              // RUNS: float4 per row
    uint32_t runs_rows;             // RUNS: rows per item (a multiple of tpw)
};

// 8-bit offset-binary levels without a table: (code - 127.5) / 35.5 in float32
// as numpy computes it (baseband/base/encoding.py:131-144).  A 256-entry table
// in shared memory suffers ~3-way bank conflicts under random codes (the LSU
// data pipe was 73 % busy); this is four ALU operations instead.
// One byte permute plants the code in the second mantissa byte of 2^23 (ulp 1:
// 2^23 + 256 code), one exact subtraction leaves x = 256 (code - 127.5), and
// the quotient is x times the reciprocal of 256 * 35.5 carried in two terms,
// hi + lo, summed in one FMA: a single rounding of a product that is exact to
// ~2^-48, which for these 256 inputs lands on the correctly rounded quotient.
// `affine8_matches` checks on the host, for all 256 codes, that this equals
// the table given (else the table path is used).
BB_HD float affine8(uint32_t w, uint32_t c) {
    const uint32_t u = byte_perm(w, 0x4B000000u, 0x7404u | (c << 4));
    const float x = add_rn(uint_as_float(u), -8421248.0f);   // 2^23 + 32640
    constexpr float r_hi = 0x1.cd8568p-14f, r_lo = 0x1.207362p-39f;
    return fma_rn(x, r_hi, mul_rn(x, r_lo));
}

inline bool affine8_matches(const float *levels) {
    for (uint32_t code = 0; code < 256; ++code) {
        const float v = affine8(code, 0);
        if (__builtin_memcmp(&v, &levels[code], 4) != 0) return false;
    }
    return true;
}

template <int BPS>
BB_HD float sint_code(uint32_t w, uint32_t pos) {
    return small_int_to_float((int32_t)(w << (32 - BPS - pos)) >> (32 - BPS));
}

// Values of codes 2j and 2j+1 of word w.
template <int BPS, int CODEC>
BB_HD F2 decode_pair(uint32_t w, uint32_t j, const float *lut) {
    F2 r;
    if (CODEC == CODEC_SINT) {
        r.x = sint_code<BPS>(w, 2 * j * BPS);
        r.y = sint_code<BPS>(w, (2 * j + 1) * BPS);
    } else if (CODEC == CODEC_AFFINE8) {
        r.x = affine8(w, 2 * j);
        r.y = affine8(w, 2 * j + 1);
    } else if (BPS <= 2) {
        uint32_t idx = (w >> (2 * BPS * j)) & ((1u << (2 * BPS)) - 1u);
        r = reinterpret_cast<const F2 *>(lut)[idx];
    } else {
        r.x = lut[(w >> (2 * j * BPS)) & ((1u << BPS) - 1u)];
        r.y = lut[(w >> ((2 * j + 1) * BPS)) & ((1u << BPS) - 1u)];
    }
    return r;
}

template <int BPS, int CODEC>
BB_HD float decode_one(uint32_t w, uint32_t c, const float *lut) {
    // one table access per value: the pair table serves 1/2 bit, wider codes
    // index the per-code table directly
    if (CODEC == CODEC_SINT) return sint_code<BPS>(w, c * BPS);
    if (CODEC == CODEC_AFFINE8) return affine8(w, c);
    if (BPS > 2) return lut[(w >> (c * BPS)) & ((1u << BPS) - 1u)];
    F2 r = decode_pair<BPS, CODEC>(w, c >> 1, lut);
    return (c & 1u) ? r.y : r.x;
}

// Register-select decode (SEL variants): the 2^BPS levels come from the
// kernel parameters (constant bank) and a value is picked with bit tests and
// selects -- no shared-memory access at all.  Only 1- and 2-bit level tables;
// `sh` is the bit position of the code in the word.
template <int BPS>
BB_HD float sel_level(uint32_t w, uint32_t sh, const LevelTable<BPS> &lv) {
    if (BPS == 1) return ((w >> sh) & 1u) ? lv.v[1] : lv.v[0];
    const bool b0 = (w >> sh) & 1u, b1 = (w >> (sh + 1u)) & 1u;
    const float lo = b0 ? lv.v[1] : lv.v[0];
    const float hi = b0 ? lv.v[3 % (1 << BPS)] : lv.v[2 % (1 << BPS)];
    return b1 ? hi : lo;
}

template <int BPS, int CODEC, bool SEL>
BB_HD F2 decode_pair_v(uint32_t w, uint32_t j, const float *lut,
                       const LevelTable<BPS> &lv) {
    if (SEL && CODEC == CODEC_LEVELS && BPS <= 2)
        return F2{sel_level<BPS>(w, 2u * j * BPS, lv),
                  sel_level<BPS>(w, (2u * j + 1u) * BPS, lv)};
    return decode_pair<BPS, CODEC>(w, j, lut);
}

template <int BPS, int CODEC, bool SEL>
BB_HD float decode_one_v(uint32_t w, uint32_t c, const float *lut,
                         const LevelTable<BPS> &lv) {
    if (SEL && CODEC == CODEC_LEVELS && BPS <= 2)
        return sel_level<BPS>(w, c * BPS, lv);
    return decode_one<BPS, CODEC>(w, c, lut);
}

BB_HD uint32_t load_u32(const uint8_t *p) {
    return *reinterpret_cast<const uint32_t *>(p);
}

// ROWGROUP: item = lw * ngroup + g, lw = word index over the launch's sets.
// Split into a fetch (address arithmetic + global loads) and an emit (decode +
// stores) so the kernel can issue the loads of several items before decoding
// the first: these kernels are latency bound otherwise.
template <int G>
struct RowItem {
    uint32_t w[G];
    uint32_t okmask;                // bit j: slot j valid
    uint32_t g, h;                  // group; which part of the word's rows
    long long row0;
    bool live;
};

// An item is at most 8 rows: a word holding more (1 and 2 bit) is split over
// SPLIT neighbouring threads, which read the same word (one broadcast load).
// Fewer stores per thread measured faster (see Unroll in bb_bitfield.cu).
template <int BPS, int G>
struct RowSplit {
    static constexpr int kTpw = (32 / BPS) / (4 / G);
    static constexpr int kRows = kTpw < 8 ? kTpw : 8;     // rows per item
    static constexpr int kSplit = kTpw / kRows;
};

template <int BPS, int G>
BB_HD void rowgroup_fetch(const DecGeom &p, uint32_t item, RowItem<G> &it) {
    constexpr int E = 4 / G;
    constexpr int TPW = (32 / BPS) / E;
    constexpr int RPI = RowSplit<BPS, G>::kRows;
    constexpr int SPLIT = RowSplit<BPS, G>::kSplit;
    uint32_t lwh, lw, set, k;
    p.div_ngroup.divmod(item, lwh, it.g);
    lw = lwh / SPLIT;
    it.h = lwh % SPLIT;
    p.div_nword.divmod(lw, set, k);
    it.row0 = p.row_base + (long long)lw * TPW + it.h * RPI;
    it.live = !(it.row0 + RPI <= 0 || it.row0 >= p.nsample);
    it.okmask = 0u;
    if (!it.live) return;
    const long long *uo = p.unit_offset + (size_t)set * p.nthread + it.g * G;
    if (p.debug) {
        // knock-out runs (tools/sweep_variants.py): 1 = no payload loads,
        // 2 = no loads at all; the words are a hash of the item
#pragma unroll
        for (int j = 0; j < G; ++j) {
            const long long off = p.debug >= 2 ? 0 : uo[j];
            it.w[j] = (item + (uint32_t)off) * 0x9E3779B1u + j;
            it.okmask |= 1u << j;
        }
        return;
    }
#pragma unroll
    for (int j = 0; j < G; ++j) {
        const long long off = uo[j];
        it.w[j] = off >= 0 ? load_u32(p.src + off + 4ull * k) : 0u;
        it.okmask |= (off >= 0 ? 1u : 0u) << j;
    }
}

template <int BPS, int CODEC, int G, bool SEL = false, typename OT = float>
BB_HD void rowgroup_emit(const DecGeom &p, const float *lut,
                         const RowItem<G> &it,
                         const LevelTable<BPS> &lv = LevelTable<BPS>()) {
    constexpr int E = 4 / G;
    constexpr int TPW = RowSplit<BPS, G>::kRows;   // rows of this item
    if (!it.live) return;
    const uint32_t c0 = it.h * TPW;                // first code (pair) used
    const uint32_t *w = it.w;
    const long long row0 = it.row0;
    const size_t rowlen = (size_t)p.nthread * E;
    OT *dst = out_as<OT>(p) + row0 * (long long)rowlen + it.g * 4;
    if (it.okmask == (1u << G) - 1u && row0 >= 0
        && row0 + TPW <= p.nsample) {
        // Fast path: all rows inside the requested range, every slot valid.
        if (E == 1) {
#pragma unroll
            for (int mm = 0; mm < TPW / 2; ++mm) {
                const uint32_t m = c0 / 2 + mm;
                F2 a = decode_pair_v<BPS, CODEC, SEL>(w[0], m, lut, lv);
                F2 b = decode_pair_v<BPS, CODEC, SEL>(w[1 % G], m, lut, lv);
                F2 c = decode_pair_v<BPS, CODEC, SEL>(w[2 % G], m, lut, lv);
                F2 d = decode_pair_v<BPS, CODEC, SEL>(w[3 % G], m, lut, lv);
                store4(dst, F4{a.x, b.x, c.x, d.x});
                dst += rowlen;
                store4(dst, F4{a.y, b.y, c.y, d.y});
                dst += rowlen;
            }
        } else {
#pragma unroll
            for (int ii = 0; ii < TPW; ++ii) {
                const uint32_t i = c0 + ii;
                F2 a = decode_pair_v<BPS, CODEC, SEL>(w[0], i, lut, lv);
                F2 b = decode_pair_v<BPS, CODEC, SEL>(w[1 % G], i, lut, lv);
                store4(dst, F4{a.x, a.y, b.x, b.y});
                dst += rowlen;
            }
        }
        return;
    }
    // Edge path: partial word at either end of the read, or invalid frames.
    const float fill_im = p.complex_fill ? 0.f : p.fill;
    const bool ok0 = it.okmask & 1u, ok1 = (it.okmask >> (1 % G)) & 1u,
        ok2 = (it.okmask >> (2 % G)) & 1u, ok3 = (it.okmask >> (3 % G)) & 1u;
#pragma unroll 1
    for (int ii = 0; ii < TPW; ++ii, dst += rowlen) {
        if (row0 + ii < 0 || row0 + ii >= p.nsample) continue;
        const uint32_t i = c0 + ii;
        F4 v;
        // (with SEL there is no table in shared memory: same select here)
        if (E == 1) {
            v.x = ok0 ? decode_one_v<BPS, CODEC, SEL>(w[0], i, lut, lv)
                : p.fill;
            v.y = ok1 ? decode_one_v<BPS, CODEC, SEL>(w[1 % G], i, lut, lv)
                : p.fill;
            v.z = ok2 ? decode_one_v<BPS, CODEC, SEL>(w[2 % G], i, lut, lv)
                : p.fill;
            v.w = ok3 ? decode_one_v<BPS, CODEC, SEL>(w[3 % G], i, lut, lv)
                : p.fill;
        } else {
            F2 a = decode_pair_v<BPS, CODEC, SEL>(w[0], i, lut, lv);
            F2 b = decode_pair_v<BPS, CODEC, SEL>(w[1 % G], i, lut, lv);
            v.x = ok0 ? a.x : p.fill;
            v.y = ok0 ? a.y : fill_im;
            v.z = ok1 ? b.x : p.fill;
            v.w = ok1 ? b.y : fill_im;
        }
        store4(dst, v);
    }
}

template <int BPS, int CODEC, int G, typename OT = float>
BB_HD void dec_rowgroup(const DecGeom &p, const float *lut, uint32_t item) {
    RowItem<G> it;
    rowgroup_fetch<BPS, G>(p, item, it);
    rowgroup_emit<BPS, CODEC, G, false, OT>(p, lut, it);
}

// RUN: item = float4 index within the launch's block of rows; again split
// into fetch and emit.
struct RunItem {
    uint32_t w, pair;               // word and first pair index within it
    long long gidx;                 // output float index, < 0: nothing to do
    bool valid;
};

template <int BPS>
BB_HD void run_fetch(const DecGeom &p, uint32_t item, RunItem &it) {
    constexpr int CPW = 32 / BPS;
    const uint32_t n = item * 4u;              // element index in the launch
    const uint32_t rowlen = p.nthread * p.nelem;
    it.gidx = p.row_base * (long long)rowlen + n;
    it.w = 0u;
    it.pair = 0u;
    it.valid = false;
    if (it.gidx < 0 || it.gidx >= p.nsample * (long long)rowlen) {
        it.gidx = -1;
        return;
    }
    uint32_t set, pcode, slot;
    if (p.nthread == 1) {
        p.div_unitlen.divmod(n, set, pcode);     // unitlen = spf * nelem
        slot = 0;
    } else {
        uint32_t row, rem, t;
        p.div_rowlen.divmod(n, row, rem);
        slot = rem >> p.log2_nelem;
        uint32_t e = rem & (p.nelem - 1u);
        p.div_spf.divmod(row, set, t);
        pcode = (t << p.log2_nelem) + e;
    }
    const long long off = p.unit_offset[(size_t)set * p.nthread + slot];
    if (off >= 0) {
        it.valid = true;
        it.w = load_u32(p.src + off + 4ull * (pcode / CPW));
        it.pair = (pcode % CPW) >> 1;
    }
}

template <int BPS, int CODEC, typename OT = float>
BB_HD void run_emit(const DecGeom &p, const float *lut, const RunItem &it) {
    if (it.gidx < 0) return;
    F4 v;
    if (it.valid) {
        F2 a = decode_pair<BPS, CODEC>(it.w, it.pair, lut);
        F2 b = decode_pair<BPS, CODEC>(it.w, it.pair + 1, lut);
        v = F4{a.x, a.y, b.x, b.y};
    } else {
        const float fill_im = p.complex_fill ? 0.f : p.fill;
        v = F4{p.fill, fill_im, p.fill, fill_im};
    }
    store4(out_as<OT>(p) + it.gidx, v);
}

template <int BPS, int CODEC, typename OT = float>
BB_HD void dec_run(const DecGeom &p, const float *lut, uint32_t item) {
    RunItem it;
    run_fetch<BPS>(p, item, it);
    run_emit<BPS, CODEC, OT>(p, lut, it);
}

// RUNS: RUN for words that hold S = tpw >= 1 complete samples of a thread slot
// (nelem * BPS * S == 32; several threads of several channels).  In RUN every
// float4 redoes two divisions, the unit-offset load and the load of a word it
// shares with S - 1 other float4 -- 93 instructions per float4, issue bound
// (profiles/r2_ncu_issue_bound_modes.txt).  Here an item is one float4
// position f of a group of R = runs_rows consecutive rows (R = max(S, 4)): the
// R float4, one per row, come out of R / S consecutive words of one slot, so
// that work is done once per R stores.  Consecutive lanes take consecutive f:
// a warp store covers whole rows (rowlen * 4 bytes each) R rows apart.  The
// planner only picks it when the read starts and ends on multiples of R rows.
struct RunsItem {
    uint32_t w[4];                  // the R / S words
    uint32_t e;                     // first element of the float4
    long long gidx;                 // output float index of row 0, < 0: none
    bool valid;
};

template <int BPS>
BB_HD void runs_fetch(const DecGeom &p, uint32_t item, RunsItem &it) {
    const uint32_t S = p.tpw, R = p.runs_rows;
    const uint32_t rowlen = p.nthread * p.nelem;
    uint32_t rg, f;
    p.div_f4row.divmod(item, rg, f);
    const uint32_t row = rg * R;                  // within the launch
    const long long row_abs = p.row_base + row;
    it.valid = false;
    it.gidx = -1;
    if (row_abs < 0 || row_abs >= p.nsample) return;
    it.gidx = row_abs * (long long)rowlen + 4ll * f;
    const uint32_t slot = (4u * f) >> p.log2_nelem;
    it.e = (4u * f) & (p.nelem - 1u);
    uint32_t set, t;
    p.div_spf.divmod(row, set, t);
    const long long off = p.unit_offset[(size_t)set * p.nthread + slot];
    if (off >= 0) {
        it.valid = true;
        const uint8_t *q = p.src + off + 4ull * (t / S);
#pragma unroll
        for (uint32_t j = 0; j < 4; ++j)
            if (j * S < R) it.w[j] = load_u32(q + 4u * j);
    }
}

template <int BPS, int CODEC, typename OT = float>
BB_HD void runs_emit(const DecGeom &p, const float *lut, const RunsItem &it) {
    if (it.gidx < 0) return;
    const uint32_t S = p.tpw, R = p.runs_rows;
    const size_t rowlen = (size_t)p.nthread * p.nelem;
    OT *dst = out_as<OT>(p) + it.gidx;
    const float fill_im = p.complex_fill ? 0.f : p.fill;
    if (!it.valid) {
        for (uint32_t r = 0; r < R; ++r, dst += rowlen)
            store4(dst, F4{p.fill, fill_im, p.fill, fill_im});
        return;
    }
#pragma unroll
    for (uint32_t j = 0; j < 4; ++j) {
        if (j * S >= R) break;
        const uint32_t w = it.w[j];
        for (uint32_t s = 0; s < S && j * S + s < R; ++s, dst += rowlen) {
            const uint32_t pair = ((s << p.log2_nelem) + it.e) >> 1;
            F2 a = decode_pair<BPS, CODEC>(w, pair, lut);
            F2 b = decode_pair<BPS, CODEC>(w, pair + 1, lut);
            store4(dst, F4{a.x, a.y, b.x, b.y});
        }
    }
}

template <int BPS, int CODEC, typename OT = float>
BB_HD void dec_runs(const DecGeom &p, const float *lut, uint32_t item) {
    RunsItem it;
    runs_fetch<BPS>(p, item, it);
    runs_emit<BPS, CODEC, OT>(p, lut, it);
}

// WORDRUN: a warp owns chunk = 32 consecutive words of the launch (nthread
// == 1, so word idx of the launch sits at float offset idx * CPW).  Phase 1:
// lane loads word chunk*32 + lane.  Phase 2 (j = 0 .. F-1, F = float4 per
// word): lane stores float4 q = lane + 32 j of the chunk, decoded from the word
// of lane wr_src_lane(lane, j), which the caller fetches with a shuffle.
template <int BPS>
BB_HD uint32_t wr_src_lane(uint32_t lane, int j) {
    constexpr int F = 8 / BPS;            // float4 per 32-bit word
    return (lane + 32u * j) / F;
}

BB_HD bool wr_load(const DecGeom &p, uint32_t chunk, uint32_t lane,
                   uint32_t &w) {
    w = 0u;
    const uint32_t idx = chunk * 32u + lane;
    if (idx >= p.nwords_total) return false;
    uint32_t unit, k;
    p.div_nword.divmod(idx, unit, k);
    const long long off = p.unit_offset[unit];
    if (off < 0) return false;
    w = load_u32(p.src + off + 4ull * k);
    return true;
}

template <int BPS, int CODEC, typename OT = float>
BB_HD void wr_emit(const DecGeom &p, const float *lut, uint32_t chunk,
                   uint32_t lane, int j, uint32_t w, bool valid) {
    constexpr int F = 8 / BPS;
    const uint32_t q = lane + 32u * j;                 // float4 in the chunk
    if (chunk * 32u + q / F >= p.nwords_total) return;
    const long long n = ((long long)chunk * (32 * F) + q) * 4;
    const long long gidx = p.row_base * (long long)p.nelem + n;
    if (gidx < 0 || gidx >= p.nsample * (long long)p.nelem) return;
    F4 v;
    if (valid) {
        const uint32_t pr = 2u * (q % F);              // first pair index
        F2 a = decode_pair<BPS, CODEC>(w, pr, lut);
        F2 b = decode_pair<BPS, CODEC>(w, pr + 1, lut);
        v = F4{a.x, a.y, b.x, b.y};
    } else {
        const float fill_im = p.complex_fill ? 0.f : p.fill;
        v = F4{p.fill, fill_im, p.fill, fill_im};
    }
    store4(out_as<OT>(p) + gidx, v);
}

// WORDROW<G, NG>: nthread * E == 4 * NG (G = 4 single-channel threads or G = 2
// threads of one complex channel per float4; NG = 1 or 2 float4 per output
// row).  Like WORDRUN, a warp takes 32 consecutive word positions -- here of
// all G * NG slots, that many coalesced 128-byte loads -- whose decoded rows
// form one contiguous run of 32 * TPW * NG float4 (TPW = rows per word).
// Store j: lane L writes float4 q = L + 32 j of the chunk = group q % NG of
// row q / NG, from the G words of that group held by lane (q / NG) / TPW
// (staged in shared memory by the kernel).  Every warp store is 512
// contiguous bytes, where ROWGROUP's would be 16 pieces of 32 bytes for rows
// of 8 floats.
template <int BPS, int G, int NG>
BB_HD uint32_t wrow_src_lane(uint32_t lane, int j) {
    return ((lane + 32u * j) / NG) / ((32 / BPS) / (4 / G));
}

// W = G * NG words (all slots of a row) of word position chunk * 32 + lane.
template <int W>
BB_HD uint32_t wrow_load(const DecGeom &p, uint32_t chunk, uint32_t lane,
                         uint32_t w[W]) {
#pragma unroll
    for (int j = 0; j < W; ++j) w[j] = 0u;
    const uint32_t idx = chunk * 32u + lane;   // word position over all sets
    if (idx >= p.nwords_total) return 0u;
    uint32_t set, k;
    p.div_nword.divmod(idx, set, k);
    const long long *uo = p.unit_offset + (size_t)set * W;
    uint32_t okmask = 0u;
#pragma unroll
    for (int j = 0; j < W; ++j) {
        const long long off = uo[j];
        if (off >= 0) {
            w[j] = load_u32(p.src + off + 4ull * k);
            okmask |= 1u << j;
        }
    }
    return okmask;
}

// One float4: code position c of the G words w; okmask bit g: slot g valid.
template <int BPS, int CODEC, int G>
BB_HD F4 wrow_decode(const DecGeom &p, const float *lut, uint32_t c,
                     const uint32_t w[G], uint32_t okmask) {
    F4 v;
    if (G == 4) {
        v = F4{decode_one<BPS, CODEC>(w[0], c, lut),
               decode_one<BPS, CODEC>(w[1 % G], c, lut),
               decode_one<BPS, CODEC>(w[2 % G], c, lut),
               decode_one<BPS, CODEC>(w[3 % G], c, lut)};
        if (okmask != 0xfu) {                      // some slot is fill
            if (!(okmask & 1u)) v.x = p.fill;
            if (!(okmask & 2u)) v.y = p.fill;
            if (!(okmask & 4u)) v.z = p.fill;
            if (!(okmask & 8u)) v.w = p.fill;
        }
    } else {
        const F2 a = decode_pair<BPS, CODEC>(w[0], c, lut);
        const F2 b = decode_pair<BPS, CODEC>(w[1 % G], c, lut);
        v = F4{a.x, a.y, b.x, b.y};
        if (okmask != 0x3u) {
            const float fill_im = p.complex_fill ? 0.f : p.fill;
            if (!(okmask & 1u)) { v.x = p.fill; v.y = fill_im; }
            if (!(okmask & 2u)) { v.z = p.fill; v.w = fill_im; }
        }
    }
    return v;
}

// Checked store (edges of the read / of the launch).  ``w`` and ``okmask``
// are those of the float4's group.
template <int BPS, int CODEC, int G, int NG, typename OT = float>
BB_HD void wrow_emit(const DecGeom &p, const float *lut, uint32_t chunk,
                     uint32_t lane, int j, const uint32_t w[G],
                     uint32_t okmask) {
    constexpr int TPW = (32 / BPS) / (4 / G);
    const uint32_t q = lane + 32u * j;                 // float4 in the chunk
    const uint32_t r = q / NG;                         // row within the chunk
    if (chunk * 32u + r / TPW >= p.nwords_total) return;
    const long long row = p.row_base + ((long long)chunk * 32 * TPW + r);
    if (row < 0 || row >= p.nsample) return;
    store4(out_as<OT>(p) + (row * NG + q % NG) * 4,
           wrow_decode<BPS, CODEC, G>(p, lut, r % TPW, w, okmask));
}

// Interior chunks (all 32 word positions inside the launch, all 32 * TPW rows
// inside the requested range; warp uniform): no per-row bounds checks, one
// 64-bit output base per chunk; the code position and the source lane are
// loop invariant per (lane, j).
template <int BPS, int G>
BB_HD bool wrow_interior(const DecGeom &p, uint32_t chunk) {
    constexpr int TPW = (32 / BPS) / (4 / G);
    if ((unsigned long long)chunk * 32u + 32u > p.nwords_total) return false;
    const long long row0 = p.row_base + (long long)chunk * (32 * TPW);
    return row0 >= 0 && row0 + 32 * TPW <= p.nsample;
}

template <int BPS, int G, int NG, typename OT = float>
BB_HD OT *wrow_chunk_out(const DecGeom &p, uint32_t chunk) {
    constexpr int TPW = (32 / BPS) / (4 / G);
    return out_as<OT>(p) + (p.row_base + (long long)chunk * (32 * TPW)) * (4 * NG);
}

template <int BPS, int CODEC, int G, int NG, typename OT>
BB_HD void wrow_emit_fast(const DecGeom &p, const float *lut, OT *chunk_out,
                          uint32_t q, const uint32_t w[G], uint32_t okmask) {
    constexpr int TPW = (32 / BPS) / (4 / G);
    store4(chunk_out + 4u * q,
           wrow_decode<BPS, CODEC, G>(p, lut, (q / NG) % TPW, w, okmask));
}

// TILE<G, P>: rows of exactly four float4 (16 single-channel threads with
// G = 4, or 8 threads of one complex channel with G = 2; NSLOT = 4 G slots):
// the headline C2 shape.  ROWGROUP's warp stores are there 8 pieces of 64
// bytes, 512 bytes apart.  Here a warp takes P consecutive word positions of
// all NSLOT slots (lane L: position L / NGR, NL = NSLOT / NGR neighbouring
// slots, NGR = 32 / P; every 32-byte sector of the packed input is used
// whole), parks the words in shared memory at word address NL * L (linear:
// conflict free) and then stores the P * TPW decoded rows as one contiguous
// run: store j, lane L writes float4 q = L + 32 j = group q % 4 of row q / 4,
// reading the G words of its group with one LDS.128 / LDS.64 (lanes of a group
// broadcast; the 4 groups of a row are 16 consecutive words).  Every store
// instruction covers 512 contiguous bytes.
template <int BPS, int G, int P>
struct Tile {
    static constexpr int kSlots = 4 * G;
    static constexpr int kNgr = 32 / P;                 // lane groups
    static constexpr int kNl = kSlots / kNgr;           // words per lane
    static constexpr int kTpw = (32 / BPS) / (4 / G);   // rows per word
    static constexpr int kStores = P * kTpw / 8;        // float4 per lane
    static constexpr int kWords = P * kSlots;           // words per chunk
};

// Words of lane `lane` of chunk `chunk`: w[i] = slot (lane % NGR) * NL + i at
// word position chunk * P + lane / NGR.  Returns the valid bits.
template <int BPS, int G, int P>
BB_HD uint32_t tile_load(const DecGeom &p, uint32_t chunk, uint32_t lane,
                         uint32_t w[Tile<BPS, G, P>::kNl]) {
    using T = Tile<BPS, G, P>;
#pragma unroll
    for (int i = 0; i < T::kNl; ++i) w[i] = 0u;
    const uint32_t idx = chunk * P + lane / T::kNgr;
    if (idx >= p.nwords_total) return 0u;
    uint32_t set, k;
    p.div_nword.divmod(idx, set, k);
    const long long *uo = p.unit_offset + (size_t)set * T::kSlots
        + (lane % T::kNgr) * T::kNl;
    uint32_t ok = 0u;
#pragma unroll
    for (int i = 0; i < T::kNl; ++i) {
        const long long off = uo[i];
        if (off >= 0) {
            w[i] = load_u32(p.src + off + 4ull * k);
            ok |= 1u << i;
        }
    }
    return ok;
}

template <int BPS, int G, int P>
BB_HD bool tile_interior(const DecGeom &p, uint32_t chunk) {
    using T = Tile<BPS, G, P>;
    if ((unsigned long long)chunk * P + P > p.nwords_total) return false;
    const long long row0 = p.row_base + (long long)chunk * (P * T::kTpw);
    return row0 >= 0 && row0 + P * T::kTpw <= p.nsample;
}

template <int BPS, int G, int P, typename OT = float>
BB_HD OT *tile_chunk_out(const DecGeom &p, uint32_t chunk) {
    using T = Tile<BPS, G, P>;
    return out_as<OT>(p) + (p.row_base + (long long)chunk * (P * T::kTpw)) * 16;
}

// float4 q of a chunk from the G words `w` of its group (all slots valid).
template <int BPS, int CODEC, int G, int P, bool SEL>
BB_HD F4 tile_decode(uint32_t q, const uint32_t w[G], const float *lut,
                     const LevelTable<BPS> &lv) {
    using T = Tile<BPS, G, P>;
    const uint32_t t = (q >> 2) % T::kTpw;          // row within the word
    if (G == 4)
        return F4{decode_one_v<BPS, CODEC, SEL>(w[0], t, lut, lv),
                  decode_one_v<BPS, CODEC, SEL>(w[1 % G], t, lut, lv),
                  decode_one_v<BPS, CODEC, SEL>(w[2 % G], t, lut, lv),
                  decode_one_v<BPS, CODEC, SEL>(w[3 % G], t, lut, lv)};
    const F2 a = decode_pair_v<BPS, CODEC, SEL>(w[0], t, lut, lv);
    const F2 b = decode_pair_v<BPS, CODEC, SEL>(w[1 % G], t, lut, lv);
    return F4{a.x, a.y, b.x, b.y};
}

// Checked store for edge chunks / chunks with invalid units.  okmask: bit s =
// slot s of the float4's group valid.
template <int BPS, int CODEC, int G, int P, bool SEL, typename OT = float>
BB_HD void tile_emit(const DecGeom &p, const float *lut,
                     const LevelTable<BPS> &lv, uint32_t chunk, uint32_t q,
                     const uint32_t w[G], uint32_t okmask) {
    using T = Tile<BPS, G, P>;
    const uint32_t r = q >> 2;                       // row within the chunk
    if (chunk * P + r / T::kTpw >= p.nwords_total) return;
    const long long row = p.row_base + (long long)chunk * (P * T::kTpw) + r;
    if (row < 0 || row >= p.nsample) return;
    F4 v = tile_decode<BPS, CODEC, G, P, SEL>(q, w, lut, lv);
    if (okmask != (1u << G) - 1u) {
        const float fill_im = p.complex_fill ? 0.f : p.fill;
        if (G == 4) {
            if (!(okmask & 1u)) v.x = p.fill;
            if (!(okmask & 2u)) v.y = p.fill;
            if (!(okmask & 4u)) v.z = p.fill;
            if (!(okmask & 8u)) v.w = p.fill;
        } else {
            if (!(okmask & 1u)) { v.x = p.fill; v.y = fill_im; }
            if (!(okmask & 2u)) { v.z = p.fill; v.w = fill_im; }
        }
    }
    store4(out_as<OT>(p) + (row * 4 + (q & 3u)) * 4, v);
}

// Valid bits of group g = q & 3 of the row of float4 q, from the per-lane
// valid bits of the whole chunk (oks[lane], bit i = word i of that lane).
template <int BPS, int G, int P>
BB_HD uint32_t tile_group_ok(const uint32_t *oks, uint32_t q) {
    using T = Tile<BPS, G, P>;
    const uint32_t pos = (q >> 2) / T::kTpw, g = q & 3u;
    uint32_t m = 0u;
#pragma unroll
    for (int s = 0; s < G; ++s) {
        const uint32_t slot = g * G + s;
        const uint32_t lane = pos * T::kNgr + slot / T::kNl;
        m |= ((oks[lane] >> (slot % T::kNl)) & 1u) << s;
    }
    return m;
}

// SCALAR: item = element index within the launch's block of rows.
template <int BPS, int CODEC, typename OT = float>
BB_HD void dec_scalar(const DecGeom &p, const float *lut, uint32_t item) {
    constexpr int CPW = 32 / BPS;
    const uint32_t rowlen = p.nthread * p.nelem;
    long long gidx = p.row_base * (long long)rowlen + item;
    if (gidx < 0 || gidx >= p.nsample * (long long)rowlen) return;
    uint32_t row, rem, slot, e, set, t;
    p.div_rowlen.divmod(item, row, rem);
    p.div_nelem.divmod(rem, slot, e);
    p.div_spf.divmod(row, set, t);
    uint32_t pcode = t * p.nelem + e;
    long long off = p.unit_offset[(size_t)set * p.nthread + slot];
    float v;
    if (off >= 0) {
        uint32_t w = load_u32(p.src + off + 4ull * (pcode / CPW));
        v = decode_one<BPS, CODEC>(w, pcode % CPW, lut);
    } else {
        v = (p.complex_fill && (e & 1u)) ? 0.f : p.fill;
    }
    store1(out_as<OT>(p) + gidx, v);
}

// ------------------------------------------------------------------ encode
struct EncGeom {
    const void *in;                 // [nset*spf][nthread][nelem] S (whole call)
    unsigned long long in_elem_offset;   // first element of this launch
    uint8_t *dst;
    const long long *unit_offset;
    uint32_t nset, nthread, nelem, nword, spf, nitems, ngroup;
    uint32_t nwords_total;          // ROWWORD: nset * nword
    int32_t log2_nelem;
    FastDiv div_nword, div_ngroup, div_nthread;
};

template <typename T> struct Vec4 {
    T x, y, z, w;
    // four consecutive values of storage type S (arith_t<S> == T)
    template <typename S>
    static BB_HD Vec4 load(const S *p) {
        T v[4];
        load4(p, v);
        return {v[0], v[1], v[2], v[3]};
    }
};

BB_HD void store_u32(uint8_t *p, uint32_t v) {
    *reinterpret_cast<uint32_t *>(p) = v;
}

template <typename S, int BPS, int QUANT, int G>
BB_HD void enc_rowgroup(const EncGeom &p, const QuantConsts<arith_t<S>> &c,
                        uint32_t item) {
    using T = arith_t<S>;
    constexpr int E = 4 / G;
    constexpr int CPW = 32 / BPS;
    constexpr int TPW = CPW / E;
    uint32_t lw, g;
    p.div_ngroup.divmod(item, lw, g);
    uint32_t set, k;
    p.div_nword.divmod(lw, set, k);
    const size_t rowlen = (size_t)p.nthread * E;
    const S *src = reinterpret_cast<const S *>(p.in) + p.in_elem_offset
        + (size_t)lw * TPW * rowlen + g * 4;
    uint32_t w[G];
#pragma unroll
    for (int j = 0; j < G; ++j) w[j] = 0u;
#pragma unroll
    for (int i = 0; i < TPW; ++i) {
        Vec4<T> v = Vec4<T>::load(src + (size_t)i * rowlen);
        uint32_t q0 = quantise<T, BPS, QUANT>(v.x, c);
        uint32_t q1 = quantise<T, BPS, QUANT>(v.y, c);
        uint32_t q2 = quantise<T, BPS, QUANT>(v.z, c);
        uint32_t q3 = quantise<T, BPS, QUANT>(v.w, c);
        if (E == 1) {
            w[0] |= q0 << (i * BPS);
            w[1 % G] |= q1 << (i * BPS);
            w[2 % G] |= q2 << (i * BPS);
            w[3 % G] |= q3 << (i * BPS);
        } else {
            w[0] |= (q0 | (q1 << BPS)) << (2 * i * BPS);
            w[1 % G] |= (q2 | (q3 << BPS)) << (2 * i * BPS);
        }
    }
    const long long *uo = p.unit_offset + (size_t)set * p.nthread + g * G;
#pragma unroll
    for (int j = 0; j < G; ++j) {
        long long off = uo[j];
        if (off >= 0) store_u32(p.dst + off + 4ull * k, w[j]);
    }
}

// ROWWORD<G>: nthread * E == 4 (4 real threads or 2 complex ones), i.e. an
// input row IS one float4 and ROWGROUP's lanes would each read their own
// 16 * TPW-byte piece (32 sectors per warp load).  Instead a warp takes the
// 32 * TPW rows behind 32 consecutive word positions: (stage) lane L loads
// rows q = L + 32 j -- every warp load is 512 contiguous bytes -- quantises
// them and parks the four codes of a row as one 32-bit value in shared
// memory; (emit) lane L collects rows L * TPW .. + TPW - 1 = its word
// position, merges them and stores one word per slot.  The XOR swizzle makes
// both the strided writes and the TPW-strided reads bank-conflict free.
template <int TPW>
BB_HD uint32_t rw_swz(uint32_t q) { return q ^ ((q >> 5) & (TPW - 1)); }

// The codes of one row: G == 4: one per byte; G == 2: (re, im) of slot 0 in
// the low half word, of slot 1 in the high one.
template <typename T, int BPS, int QUANT, int G>
BB_HD uint32_t rw_pack_row(const Vec4<T> &v, const QuantConsts<T> &c) {
    const uint32_t q0 = quantise<T, BPS, QUANT>(v.x, c),
        q1 = quantise<T, BPS, QUANT>(v.y, c),
        q2 = quantise<T, BPS, QUANT>(v.z, c),
        q3 = quantise<T, BPS, QUANT>(v.w, c);
    if (G == 4) return q0 | (q1 << 8) | (q2 << 16) | (q3 << 24);
    return (q0 | (q1 << BPS)) | ((q2 | (q3 << BPS)) << 16);
}

template <typename S, int BPS, int QUANT, int G>
BB_HD void rw_stage(const EncGeom &p, const QuantConsts<arith_t<S>> &c,
                    uint32_t chunk, uint32_t lane, uint32_t *buf) {
    using T = arith_t<S>;
    constexpr int TPW = (32 / BPS) / (4 / G);
    constexpr int LB = TPW < 8 ? TPW : 8;         // loads in flight per lane
    const size_t nrows = (size_t)p.nwords_total * TPW;
    const size_t row0 = (size_t)chunk * (32 * TPW);
    const S *in = reinterpret_cast<const S *>(p.in) + p.in_elem_offset;
#pragma unroll
    for (int j0 = 0; j0 < TPW; j0 += LB) {
        Vec4<T> v[LB];
#pragma unroll
        for (int j = 0; j < LB; ++j) {
            const size_t row = row0 + lane + 32u * (j0 + j);
            if (row < nrows) v[j] = Vec4<T>::load(in + row * 4);
            else v[j] = Vec4<T>{(T)0, (T)0, (T)0, (T)0};
        }
#pragma unroll
        for (int j = 0; j < LB; ++j)
            buf[rw_swz<TPW>(lane + 32u * (j0 + j))] =
                rw_pack_row<T, BPS, QUANT, G>(v[j], c);
    }
}

template <int BPS, int G>
BB_HD void rw_emit(const EncGeom &p, uint32_t chunk, uint32_t lane,
                   const uint32_t *buf) {
    constexpr int E = 4 / G;
    constexpr int TPW = (32 / BPS) / E;
    constexpr int NC = E == 1 ? 4 : 2;            // merged values per word set
    constexpr int PER = TPW / NC;                 // rows merged into each
    const uint32_t idx = chunk * 32u + lane;      // word position, all sets
    if (idx >= p.nwords_total) return;
    uint32_t m[NC];
#pragma unroll
    for (int n = 0; n < NC; ++n) {
        m[n] = 0u;
#pragma unroll
        for (int r = 0; r < PER; ++r)
            m[n] |= buf[rw_swz<TPW>(lane * TPW + n * PER + r)]
                << (r * BPS * E);
    }
    uint32_t w[G];
    if (G == 4) {                                 // 4 x 4 byte transpose
        const uint32_t lo01 = byte_perm(m[0], m[1 % NC], 0x5140),
            lo23 = byte_perm(m[2 % NC], m[3 % NC], 0x5140),
            hi01 = byte_perm(m[0], m[1 % NC], 0x7362),
            hi23 = byte_perm(m[2 % NC], m[3 % NC], 0x7362);
        w[0] = byte_perm(lo01, lo23, 0x5410);
        w[1 % G] = byte_perm(lo01, lo23, 0x7632);
        w[2 % G] = byte_perm(hi01, hi23, 0x5410);
        w[3 % G] = byte_perm(hi01, hi23, 0x7632);
    } else {
        w[0] = byte_perm(m[0], m[1 % NC], 0x5410);
        w[1 % G] = byte_perm(m[0], m[1 % NC], 0x7632);
    }
    uint32_t set, k;
    p.div_nword.divmod(idx, set, k);
    const long long *uo = p.unit_offset + (size_t)set * G;
#pragma unroll
    for (int j = 0; j < G; ++j) {
        const long long off = uo[j];
        if (off >= 0) store_u32(p.dst + off + 4ull * k, w[j]);
    }
}

// Vectorised word encode split into fetch (addresses + float4 loads) and
// emit (quantise, pack, store) so a kernel can have the loads of several words
// in flight (8- and 4-bit words need only one or two float4 each).
template <typename T, int BPS>
struct EncWordItem {
    Vec4<T> v[(32 / BPS) / 4];
    uint8_t *dst;                   // null: nothing to do
};

template <typename S, int BPS>
BB_HD void enc_word_fetch(const EncGeom &p, uint32_t item,
                          EncWordItem<arith_t<S>, BPS> &it) {
    using T = arith_t<S>;
    constexpr int CPW = 32 / BPS;
    uint32_t rest, k, set, slot;
    p.div_nthread.divmod(item, rest, slot);
    p.div_nword.divmod(rest, set, k);
    const long long off = p.unit_offset[set * p.nthread + slot];
    it.dst = nullptr;
    if (off < 0) return;
    it.dst = p.dst + off + 4ull * k;
    const S *in = reinterpret_cast<const S *>(p.in) + p.in_elem_offset;
    const size_t rowlen = (size_t)p.nthread * p.nelem;
    const size_t set_base = (size_t)set * p.spf * rowlen;
#pragma unroll
    for (int m = 0; m < CPW / 4; ++m) {
        const uint32_t pc = k * CPW + 4 * m;
        size_t idx;
        if (p.nthread == 1) {
            idx = set_base + pc;
        } else {
            const uint32_t t = pc >> p.log2_nelem, e = pc & (p.nelem - 1u);
            idx = set_base + ((size_t)t * p.nthread + slot) * p.nelem + e;
        }
        it.v[m] = Vec4<T>::load(in + idx);
    }
}

template <typename T, int BPS, int QUANT>
BB_HD void enc_word_emit(const QuantConsts<T> &c,
                         const EncWordItem<T, BPS> &it) {
    constexpr int CPW = 32 / BPS;
    if (it.dst == nullptr) return;
    uint32_t w = 0u;
#pragma unroll
    for (int m = 0; m < CPW / 4; ++m) {
        const uint32_t f = quantise<T, BPS, QUANT>(it.v[m].x, c)
            | (quantise<T, BPS, QUANT>(it.v[m].y, c) << BPS)
            | (quantise<T, BPS, QUANT>(it.v[m].z, c) << (2 * BPS))
            | (quantise<T, BPS, QUANT>(it.v[m].w, c) << (3 * BPS));
        w |= f << (4 * m * BPS);
    }
    store_u32(it.dst, w);
}

// RUNQ (8 bit): item = four consecutive words of one unit = 16 codes of one
// row segment; `div_nword` divides by the number of such quads per unit.
template <typename T>
struct EncQuadItem {
    Vec4<T> v[4];
    uint8_t *dst;                   // null: nothing to do
};

template <typename S>
BB_HD void enc_quad_fetch(const EncGeom &p, uint32_t item,
                          EncQuadItem<arith_t<S>> &it) {
    using T = arith_t<S>;
    uint32_t rest, kq, set, slot;
    p.div_nthread.divmod(item, rest, slot);
    p.div_nword.divmod(rest, set, kq);
    const long long off = p.unit_offset[set * p.nthread + slot];
    it.dst = nullptr;
    if (off < 0) return;
    it.dst = p.dst + off + 16ull * kq;
    const S *in = reinterpret_cast<const S *>(p.in) + p.in_elem_offset;
    const size_t rowlen = (size_t)p.nthread * p.nelem;
    const uint32_t pc = kq * 16u;
    size_t idx = (size_t)set * p.spf * rowlen;
    if (p.nthread == 1) {
        idx += pc;
    } else {
        const uint32_t t = pc >> p.log2_nelem, e = pc & (p.nelem - 1u);
        idx += ((size_t)t * p.nthread + slot) * p.nelem + e;
    }
#pragma unroll
    for (int m = 0; m < 4; ++m) it.v[m] = Vec4<T>::load(in + idx + 4 * m);
}

template <typename T, int QUANT>
BB_HD void enc_quad_emit(const QuantConsts<T> &c, const EncQuadItem<T> &it) {
    if (it.dst == nullptr) return;
    uint32_t w[4];
#pragma unroll
    for (int m = 0; m < 4; ++m)
        w[m] = quantise<T, 8, QUANT>(it.v[m].x, c)
            | (quantise<T, 8, QUANT>(it.v[m].y, c) << 8)
            | (quantise<T, 8, QUANT>(it.v[m].z, c) << 16)
            | (quantise<T, 8, QUANT>(it.v[m].w, c) << 24);
    if ((reinterpret_cast<uintptr_t>(it.dst) & 15u) == 0) {
        *reinterpret_cast<U4 *>(it.dst) = U4{w[0], w[1], w[2], w[3]};
    } else {
#pragma unroll
        for (int m = 0; m < 4; ++m) store_u32(it.dst + 4 * m, w[m]);
    }
}

// RUN / SCALAR: item = output word index over all units of the launch.
template <typename S, int BPS, int QUANT, bool VEC>
BB_HD void enc_word(const EncGeom &p, const QuantConsts<arith_t<S>> &c,
                    uint32_t item) {
    using T = arith_t<S>;
    constexpr int CPW = 32 / BPS;
    // item = (set, k, slot), slot fastest: neighbouring lanes read the slots
    // of the same rows, i.e. neighbouring bytes of the input.
    uint32_t rest, k, set, slot;
    p.div_nthread.divmod(item, rest, slot);
    p.div_nword.divmod(rest, set, k);
    const uint32_t unit = set * p.nthread + slot;
    long long off = p.unit_offset[unit];
    if (off < 0) return;
    const S *in = reinterpret_cast<const S *>(p.in) + p.in_elem_offset;
    const size_t rowlen = (size_t)p.nthread * p.nelem;
    const size_t set_base = (size_t)set * p.spf * rowlen;
    uint32_t w = 0u;
    if (VEC) {
        EncWordItem<T, BPS> it;
        enc_word_fetch<S, BPS>(p, item, it);
        enc_word_emit<T, BPS, QUANT>(c, it);
        return;
    } else {
        for (int i = 0; i < CPW; ++i) {
            uint32_t pc = k * CPW + i;
            uint32_t t = pc / p.nelem, e = pc % p.nelem;
            size_t idx = set_base + ((size_t)t * p.nthread + slot) * p.nelem + e;
            w |= quantise<T, BPS, QUANT>(widen(in[idx]), c) << (i * BPS);
        }
    }
    store_u32(p.dst + off + 4ull * k, w);
}

}  // namespace bb
