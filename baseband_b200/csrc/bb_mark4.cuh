// Mark 4 track-word codec: per-thread bodies (host/device).
//
// A frame is 20000 time steps of one ntrack-bit little-endian word; the first
// 160 steps hold the header, so the first 160*fanout samples of every frame
// decode to fill_value (baseband/mark4/frame.py:185-189, :253-258).  A payload
// word holds fanout consecutive samples of nchan channels as (sign, magnitude)
// bit pairs scattered over the tracks (SURVEY.md appendix A).
//
//  FAST     standard fan-out 4 layouts with 32 or 64 tracks (4 or 8 channels;
//           C3).  Each 32-bit half word carries 4 channels x 4 samples.  The
//           reference's `reorder32/64` bit swap (mark4/payload.py:48-69) is
//           applied in registers; afterwards byte perm[c] holds channel c as
//           four 2-bit codes (sign | magnitude << 1), which is exactly the
//           pair-LUT layout of the VDIF kernel.  A thread decodes one half
//           word into four float4 rows.
//  GENERIC  any of the five modes, table driven: bit position of sign and
//           magnitude for every (sample-in-word, channel).  Output-centric
//           float4 (or scalar) items.
#pragma once
#include "bb_common.cuh"
#include "bb_quant.cuh"

namespace bb {

struct M4Geom {
    const uint8_t *src;              // decode input / encode output base
    const long long *unit_offset;    // per frame payload offset; null => 0
    void *out;                       // decode output (row 0 of the call;
                                     // float32, F16 or BF16 elements)
    const void *in;                  // encode input
    unsigned long long in_elem_offset;
    long long row_base, nsample;
    uint32_t nframe, nchan, fanout, wordbytes, nitems;
    uint32_t steps;                  // time steps per frame (20000) or nword
    uint32_t header_steps;           // 160, or 0 for bare payload words
    int32_t log2_nchan;
    float fill;
    FastDiv div_steps, div_spf;
    uint16_t pos[32];                // sign bit | magnitude bit << 8
    float levels[4];                 // indexed 2*sign + magnitude
    // WARP mode: the launch seen as 32-bit values, frame after frame
    uint32_t per_frame32, total32;   // values per frame / in the launch
    int32_t log2_wordbytes;
    uint8_t psel[8];                 // 64-track: float4 positions of half 0, 1
    FastDiv div_frame32;
    uint32_t std4;                   // WARP mode: standard fan-out 4 fast decode
};

BB_HD uint32_t m4_reorder32(uint32_t x) {
    return (x & 0xAA55AA55u) | ((x & 0x55005500u) >> 7)
        | ((x & 0x00AA00AAu) << 7);
}

// Pair LUT as DecodeLut<2> builds it from levels indexed by the raw 2-bit
// code (sign | magnitude << 1): idx = nibble -> (value of low code, high code)
BB_HD F2 m4_pair(uint32_t byte_, uint32_t fp, const float *lut) {
    return reinterpret_cast<const F2 *>(lut)[(byte_ >> (4 * fp)) & 15u];
}

// FAST decode.  item = (frame, step, half).
template <typename OT = float>
BB_HD void m4_dec_fast(const M4Geom &p, const float *lut, uint32_t item) {
    const uint32_t nhalf = p.wordbytes >> 2;           // 1 or 2
    const uint32_t h = item & (nhalf - 1u);
    const uint32_t fs = nhalf == 2 ? item >> 1 : item;
    uint32_t frame, step;
    p.div_steps.divmod(fs, frame, step);
    const long long row0 = p.row_base
        + ((long long)frame * p.steps + step) * 4;
    if (row0 + 4 <= 0 || row0 >= p.nsample) return;
    const long long off = p.unit_offset ? p.unit_offset[frame] : 0;
    const bool data = off >= 0 && step >= p.header_steps;
    OT *dst = out_as<OT>(p) + row0 * (long long)p.nchan + 4 * h;
    F4 rows[4];
    if (data) {
        uint32_t w = *reinterpret_cast<const uint32_t *>(
            p.src + off + (size_t)(step - p.header_steps) * p.wordbytes
            + 4 * h);
        uint32_t r = m4_reorder32(w);
        uint32_t b0 = r & 0xffu, b1 = (r >> 16) & 0xffu,   // perm 0,2,1,3
            b2 = (r >> 8) & 0xffu, b3 = r >> 24;
#pragma unroll
        for (int fp = 0; fp < 2; ++fp) {
            F2 a = m4_pair(b0, fp, lut), b = m4_pair(b1, fp, lut),
                c = m4_pair(b2, fp, lut), d = m4_pair(b3, fp, lut);
            rows[2 * fp] = F4{a.x, b.x, c.x, d.x};
            rows[2 * fp + 1] = F4{a.y, b.y, c.y, d.y};
        }
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) rows[i] = F4{p.fill, p.fill, p.fill, p.fill};
    }
    if (row0 >= 0 && row0 + 4 <= p.nsample) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            store4(dst + (size_t)i * p.nchan, rows[i]);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (row0 + i >= 0 && row0 + i < p.nsample)
                store4(dst + (long long)i * p.nchan, rows[i]);
    }
}

BB_HD unsigned long long m4_load_word(const uint8_t *p, uint32_t wordbytes) {
    if (wordbytes == 8) return *reinterpret_cast<const unsigned long long *>(p);
    if (wordbytes == 4) return *reinterpret_cast<const uint32_t *>(p);
    if (wordbytes == 2) return *reinterpret_cast<const uint16_t *>(p);
    return *p;
}

BB_HD float m4_value(const M4Geom &p, unsigned long long w, uint32_t f,
                     uint32_t c) {
    uint32_t pp = p.pos[(f << p.log2_nchan) + c];
    uint32_t s = (uint32_t)(w >> (pp & 0xffu)) & 1u;
    uint32_t m = (uint32_t)(w >> (pp >> 8)) & 1u;
    return p.levels[2 * s + m];
}

// GENERIC decode of one output element (row_local, c) of the launch.
BB_HD float m4_dec_element(const M4Geom &p, uint32_t row_local, uint32_t c) {
    uint32_t frame, t;
    p.div_spf.divmod(row_local, frame, t);
    const long long off = p.unit_offset ? p.unit_offset[frame] : 0;
    const uint32_t step = t / p.fanout, f = t % p.fanout;
    if (off < 0 || step < p.header_steps) return p.fill;
    unsigned long long w = m4_load_word(
        p.src + off + (size_t)(step - p.header_steps) * p.wordbytes,
        p.wordbytes);
    return m4_value(p, w, f, c);
}

template <bool VEC, typename OT = float>
BB_HD void m4_dec_generic(const M4Geom &p, uint32_t item) {
    const uint32_t n = VEC ? item * 4u : item;
    long long gidx = p.row_base * (long long)p.nchan + n;
    if (gidx < 0 || gidx >= p.nsample * (long long)p.nchan) return;
    if (VEC) {
        float v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            uint32_t e = n + i;
            v[i] = m4_dec_element(p, e >> p.log2_nchan, e & (p.nchan - 1u));
        }
        store4(out_as<OT>(p) + gidx, F4{v[0], v[1], v[2], v[3]});
    } else {
        store1(out_as<OT>(p) + gidx,
               m4_dec_element(p, n >> p.log2_nchan, n & (p.nchan - 1u)));
    }
}

// WARP decode, every layout.  A track word of W bytes decodes to W float4
// that are contiguous in the output, so the launch is one flat run: a warp
// loads 32 consecutive 32-bit values (128 B coalesced) = 128 float4 of
// output and each lane stores float4 q = lane + 32 j (j = 0..3) -- 512
// contiguous bytes per store instruction -- fetching the 32-bit value that
// holds its four (sign, magnitude) pairs from another lane by shuffle.  The
// bit positions come from the same table as the GENERIC path (staged in shared
// memory); all eight bits of a float4 lie in one 32-bit half for the five
// supported layouts (checked by the planner).
BB_HD bool m4w_load(const M4Geom &p, uint32_t chunk, uint32_t lane,
                    uint32_t &w) {
    w = 0u;
    const uint32_t g32 = chunk * 32u + lane;
    if (g32 >= p.total32) return false;
    uint32_t frame, i32;
    p.div_frame32.divmod(g32, frame, i32);
    const long long off = p.unit_offset ? p.unit_offset[frame] : 0;
    const uint32_t step = (i32 * 4u) >> p.log2_wordbytes;
    if (off < 0 || step < p.header_steps) return false;
    w = *reinterpret_cast<const uint32_t *>(
        p.src + off - (long long)p.header_steps * p.wordbytes + 4ull * i32);
    return true;
}

// Since the word size W divides 32, float4 q = lane + 32 j sits at the same
// position q % W of its track word for every j: the eight bit positions a
// lane needs are loop invariant.
struct M4Lane {
    uint32_t sbit[4], mbit[4];      // shifts inside the 32-bit value
    uint32_t half;                  // which 32-bit half of a 64-track word
};

BB_HD M4Lane m4w_lane(const M4Geom &p, const uint16_t *pos, uint32_t lane) {
    M4Lane c;
    const uint32_t pp = lane & (p.wordbytes - 1u);     // float4 within word
    // 16-track words: two words share a 32-bit value
    const uint32_t base = (((lane >> p.log2_wordbytes) << p.log2_wordbytes)
                           & 3u) * 8u;
    c.half = (pos[4u * pp] & 0xffu) >> 5;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t sm = pos[4u * pp + k];
        c.sbit[k] = ((sm & 0xffu) & 31u) + base;
        c.mbit[k] = ((sm >> 8) & 31u) + base;
    }
    return c;
}

// Lane (within the chunk) holding the bits of float4 q of the chunk.
BB_HD uint32_t m4w_src_lane(const M4Geom &p, const M4Lane &c, uint32_t q) {
    const uint32_t n = q >> p.log2_wordbytes;          // track word in chunk
    return ((n << p.log2_wordbytes) >> 2) + c.half;
}

template <typename OT = float>
BB_HD void m4w_emit(const M4Geom &p, const M4Lane &c, const float lv[4],
                    uint32_t chunk, uint32_t q, uint32_t w, bool valid) {
    if (chunk * 32u + m4w_src_lane(p, c, q) >= p.total32) return;
    const long long gidx = p.row_base * (long long)p.nchan
        + ((long long)chunk * 128 + q) * 4;
    if (gidx < 0 || gidx >= p.nsample * (long long)p.nchan) return;
    F4 v;
    if (valid) {
        float e[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool sb = (w >> c.sbit[k]) & 1u, mb = (w >> c.mbit[k]) & 1u;
            e[k] = sb ? (mb ? lv[3] : lv[2]) : (mb ? lv[1] : lv[0]);
        }
        v = F4{e[0], e[1], e[2], e[3]};
    } else {
        v = F4{p.fill, p.fill, p.fill, p.fill};
    }
    store4(out_as<OT>(p) + gidx, v);
}

// Interior chunks (all 32 values inside the launch, all 128 float4 inside the
// requested rows; warp uniform): no per-float4 bounds checks, one 64-bit
// output base per chunk, and the levels come from the pair table of the FAST
// path (index = s0 | m0 << 1 | s1 << 2 | m1 << 3 -> two floats per LDS.64).
BB_HD bool m4w_interior(const M4Geom &p, uint32_t chunk) {
    if ((unsigned long long)chunk * 32u + 32u > p.total32) return false;
    const long long g0 = p.row_base * (long long)p.nchan
        + (long long)chunk * 512;
    return g0 >= 0 && g0 + 512 <= p.nsample * (long long)p.nchan;
}

template <typename OT = float>
BB_HD OT *m4w_chunk_out(const M4Geom &p, uint32_t chunk) {
    return out_as<OT>(p) + (p.row_base * (long long)p.nchan + (long long)chunk * 512);
}

BB_HD uint32_t m4w_pair_index(const M4Lane &c, uint32_t w, int k) {
    return ((w >> c.sbit[k]) & 1u) | (((w >> c.mbit[k]) & 1u) << 1)
        | (((w >> c.sbit[k + 1]) & 1u) << 2)
        | (((w >> c.mbit[k + 1]) & 1u) << 3);
}

template <typename OT>
BB_HD void m4w_emit_fast(const M4Geom &p, const M4Lane &c, const float *lut,
                         OT *chunk_out, uint32_t q, uint32_t w, bool valid) {
    F4 v;
    if (valid) {
        const F2 a = reinterpret_cast<const F2 *>(lut)[m4w_pair_index(c, w, 0)];
        const F2 b = reinterpret_cast<const F2 *>(lut)[m4w_pair_index(c, w, 2)];
        v = F4{a.x, a.y, b.x, b.y};
    } else {
        v = F4{p.fill, p.fill, p.fill, p.fill};
    }
    store4(chunk_out + 4u * q, v);
}

// WARP decode specialised for the standard fan-out 4 layouts (32 and 64
// tracks; C3): after `reorder32` (done once per loaded value, before the
// shuffle) byte perm[c] of a 32-bit value holds channel c as four 2-bit codes,
// so row i of its four channels is two pair-table look-ups -- no per-bit
// extraction.  float4 q of a chunk is row i of value src: 64 tracks (8
// channels, two values per track word): i = (q % 8) / 2, half q % 2; 32
// tracks: i = q % 4.
BB_HD uint32_t m4s_row(const M4Geom &p, uint32_t q) {
    const uint32_t pp = q & (p.wordbytes - 1u);
    return p.wordbytes == 8 ? pp >> 1 : pp;
}

BB_HD uint32_t m4s_src_lane(const M4Geom &p, uint32_t q) {
    const uint32_t n = q >> p.log2_wordbytes;          // track word in chunk
    return ((n << p.log2_wordbytes) >> 2)
        + (p.wordbytes == 8 ? (q & 1u) : 0u);
}

BB_HD F4 m4s_decode(uint32_t r, uint32_t i, const float *lut) {
    const uint32_t x = r >> (2u * i);
    const F2 a = reinterpret_cast<const F2 *>(lut)[
        (x & 3u) | ((x >> 14) & 12u)];                 // bytes 0, 2: ch 0, 1
    const F2 b = reinterpret_cast<const F2 *>(lut)[
        ((x >> 8) & 3u) | ((x >> 22) & 12u)];          // bytes 1, 3: ch 2, 3
    return F4{a.x, a.y, b.x, b.y};
}

template <typename OT>
BB_HD void m4s_emit_fast(const M4Geom &p, const float *lut, OT *chunk_out,
                         uint32_t q, uint32_t i, uint32_t r, bool valid) {
    store4(chunk_out + 4u * q, valid
           ? m4s_decode(r, i, lut) : F4{p.fill, p.fill, p.fill, p.fill});
}

// ------------------------------------------------------------------ encode
// FAST encode: item = (frame, step, half); header steps are skipped.  The
// encoders read storage type S and quantise in arith_t<S> (bb_common.cuh).
template <typename S>
BB_HD void m4_enc_fast(const M4Geom &p, const QuantConsts<arith_t<S>> &c,
                       uint32_t item) {
    using T = arith_t<S>;
    const uint32_t nhalf = p.wordbytes >> 2;
    const uint32_t h = item & (nhalf - 1u);
    const uint32_t fs = nhalf == 2 ? item >> 1 : item;
    uint32_t frame, step;
    p.div_steps.divmod(fs, frame, step);
    const long long off = p.unit_offset ? p.unit_offset[frame] : 0;
    if (off < 0 || step < p.header_steps) return;
    const S *src = reinterpret_cast<const S *>(p.in) + p.in_elem_offset
        + (((size_t)frame * p.steps + step) * 4) * p.nchan + 4 * h;
    uint32_t bytes[4] = {0u, 0u, 0u, 0u};       // per channel j of this half
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        T v[4];
        load4(src + (size_t)f * p.nchan, v);
#pragma unroll
        for (int j = 0; j < 4; ++j)             // raw code = sign | mag << 1
            bytes[j] |= quantise<T, 2, QUANT_MARK5B>(v[j], c) << (2 * f);
    }
    // channel j lives in byte perm[j] = {0, 2, 1, 3} before the bit reorder
    uint32_t r = bytes[0] | (bytes[1] << 16) | (bytes[2] << 8)
        | (bytes[3] << 24);
    *reinterpret_cast<uint32_t *>(const_cast<uint8_t *>(p.src) + off
        + (size_t)(step - p.header_steps) * p.wordbytes + 4 * h)
        = m4_reorder32(r);
}

// GENERIC encode: item = (frame, step) -> one whole track word.
template <typename S>
BB_HD void m4_enc_generic(const M4Geom &p, const QuantConsts<arith_t<S>> &c,
                          uint32_t item) {
    using T = arith_t<S>;
    uint32_t frame, step;
    p.div_steps.divmod(item, frame, step);
    const long long off = p.unit_offset ? p.unit_offset[frame] : 0;
    if (off < 0 || step < p.header_steps) return;
    const S *src = reinterpret_cast<const S *>(p.in) + p.in_elem_offset
        + (((size_t)frame * p.steps + step) * p.fanout) * p.nchan;
    unsigned long long w = 0ull;
    const uint32_t nval = p.fanout * p.nchan;
    for (uint32_t i = 0; i < nval; ++i) {
        uint32_t q = quantise<T, 2, QUANT_OFFSET>(widen(src[i]), c);   // 2*s + m
        uint32_t pp = p.pos[i];
        w |= (unsigned long long)(q >> 1) << (pp & 0xffu);
        w |= (unsigned long long)(q & 1u) << (pp >> 8);
    }
    uint8_t *dst = const_cast<uint8_t *>(p.src) + off
        + (size_t)(step - p.header_steps) * p.wordbytes;
    if (p.wordbytes == 8) *reinterpret_cast<unsigned long long *>(dst) = w;
    else if (p.wordbytes == 4) *reinterpret_cast<uint32_t *>(dst) = (uint32_t)w;
    else *reinterpret_cast<uint16_t *>(dst) = (uint16_t)w;
}

// HALF encode, every layout: a thread produces one 32-bit value of the track
// stream (item = value index over the launch, frames laid end to end).  Its 16
// samples are four float4 of the input -- contiguous for 16/32-track words,
// 32 bytes apart for the 64-track layouts -- loaded as vectors; sign and
// magnitude bits are placed with the per-layout table.  Stores are 128
// contiguous bytes per warp.
// The bit positions a thread needs depend only on the layout and, for 64-track
// words, on which 32-bit half the value is (h = value index & 1; the number of
// values per frame is even, so h is the parity of the item): they are turned
// into 16 sign masks and 16 magnitude masks once per thread, and a sample
// then costs three compares and two predicated ORs.
struct M4HalfMasks {
    uint32_t s[16], m[16];           // [4 * float4 + element]
    uint32_t pps[4];                 // float4 position in the track word
};

template <int W>
BB_HD M4HalfMasks m4_half_masks(const M4Geom &p, const uint16_t *pos,
                                uint32_t h) {
    M4HalfMasks mk;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        mk.pps[m] = W == 2 ? (m & 1u) : W == 4 ? (uint32_t)m
                                               : (uint32_t)p.psel[4u * h + m];
        const uint32_t base = W == 2 ? 16u * (m >> 1) : 0u;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t sm = pos[4u * mk.pps[m] + k];
            mk.s[4 * m + k] = 1u << (((sm & 0xffu) & 31u) + base);
            mk.m[4 * m + k] = 1u << (((sm >> 8) & 31u) + base);
        }
    }
    return mk;
}

template <typename S, int W>
BB_HD void m4_enc_half_w(const M4Geom &p, const M4HalfMasks &mk,
                         const QuantConsts<arith_t<S>> &c, uint32_t item) {
    using T = arith_t<S>;
    if (item >= p.total32) return;
    uint32_t frame, i32;
    p.div_frame32.divmod(item, frame, i32);
    const long long off = p.unit_offset ? p.unit_offset[frame] : 0;
    const uint32_t step = W == 8 ? i32 >> 1 : W == 4 ? i32 : i32 << 1;
    if (off < 0 || step < p.header_steps) return;
    // first track word of this value, counted over the launch
    const size_t word0 = (size_t)frame * p.steps + step;
    const S *in = reinterpret_cast<const S *>(p.in) + p.in_elem_offset;
    T v[4][4];
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        // m-th float4 of this value: (word, position in word)
        const uint32_t wsel = W == 2 ? (m >> 1) : 0u;
        load4(in + ((word0 + wsel) * W + mk.pps[m]) * 4, v[m]);
    }
    uint32_t out = 0u;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            // code = (v >= x1) + (v >= x2) + (v >= x3) (quant2_offset); its
            // high bit is the sign, its low bit the magnitude
            const T x = v[m][k];
            const bool sign = x >= c.x2;
            const bool mag = (x >= c.x3) | ((x >= c.x1) & !sign);
            out |= sign ? mk.s[4 * m + k] : 0u;
            out |= mag ? mk.m[4 * m + k] : 0u;
        }
    }
    *reinterpret_cast<uint32_t *>(const_cast<uint8_t *>(p.src) + off
        - (long long)p.header_steps * W + 4ull * i32) = out;
}

// Per-item form (masks rebuilt for every value): the CPU emulation.
template <typename S>
BB_HD void m4_enc_half(const M4Geom &p, const uint16_t *pos,
                       const QuantConsts<arith_t<S>> &c, uint32_t item) {
    if (p.wordbytes == 8)
        m4_enc_half_w<S, 8>(p, m4_half_masks<8>(p, pos, item & 1u), c, item);
    else if (p.wordbytes == 4)
        m4_enc_half_w<S, 4>(p, m4_half_masks<4>(p, pos, 0u), c, item);
    else
        m4_enc_half_w<S, 2>(p, m4_half_masks<2>(p, pos, 0u), c, item);
}

}  // namespace bb
