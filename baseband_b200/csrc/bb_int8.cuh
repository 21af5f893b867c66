// int8 <-> float32 with a 2-D transpose through a shared-memory tile.
//
// GUPPI channels-first payloads are stored [chan][time][pol][re,im] and decode
// to (time, pol, chan) (baseband/guppi/payload.py:90-110); MKBF DADA heaps are
// stored [pol][chan][256 times][re,im] and decode to (time, pol, chan)
// (baseband/dada/payload.py:54-89).  Both are
//     in  unit: [nrow][ncol] items of IB bytes (1 real, 2 complex)
//     out     : [column][nrow] items -> IB floats each
// A CTA moves one TR x TC tile: rows are read with coalesced 4-byte loads
// into shared memory (row pitch padded by one word -> conflict-free column
// reads), then written so that consecutive lanes cover consecutive rows of
// one output column = contiguous floats in HBM.
//
// Written as two per-thread phases separated by a CTA barrier so the CPU
// emulation can run them as two loops.
#pragma once
#include "bb_common.cuh"
#include "bb_quant.cuh"

namespace bb {

constexpr int kI8Rows = 32;            // tile rows (channels)
constexpr int kI8RowBytes = 128;       // tile row width in bytes
constexpr int kI8Pitch = kI8RowBytes + 4;
constexpr int kI8Threads = 256;
constexpr int kI8SmemBytes = kI8Rows * kI8Pitch;

struct I8Geom {
    const uint8_t *src;              // decode: packed input; encode: output
    const long long *unit_offset;    // [nunit]
    const long long *col_begin, *col_end, *out_col0;   // decode only
    void *out;                       // float32, F16 or BF16 elements
    const void *in;                  // encode input (float, double, F16, BF16)
    uint32_t nunit, nrow, ncol, ib;  // ib = item bytes (1 or 2)
    uint32_t tiles_r, tiles_c;       // tiles per unit
    uint32_t group;                  // fast path: column tiles per group
    uint32_t knock;                  // experiments: 1 no loads, 2 no stores
};

struct I8Tile { uint32_t unit, r0, j0; };

BB_HD I8Tile i8_tile(const I8Geom &p, uint32_t block) {
    I8Tile t;
    uint32_t per_unit = p.tiles_r * p.tiles_c;
    t.unit = block / per_unit;
    uint32_t rem = block - t.unit * per_unit;
    uint32_t tr = rem / p.tiles_c;
    t.r0 = tr * kI8Rows;
    t.j0 = (rem - tr * p.tiles_c) * (kI8RowBytes / p.ib);
    return t;
}

// Phase 1 of decode: packed rows -> shared tile.
BB_HD void i8_dec_load(const I8Geom &p, uint8_t *smem, uint32_t block,
                       uint32_t tid) {
    I8Tile t = i8_tile(p, block);
    const long long off = p.unit_offset[t.unit];
    if (off < 0) return;
    if ((long long)t.j0 >= p.col_end[t.unit]
        || (long long)t.j0 + kI8RowBytes / p.ib <= p.col_begin[t.unit]) return;
    const uint32_t lane = tid & 31u, warp = tid >> 5;
    const size_t rowbytes = (size_t)p.ncol * p.ib;
    const size_t b0 = (size_t)t.j0 * p.ib + 4 * lane;     // byte within row
    for (uint32_t r = warp; r < kI8Rows; r += kI8Threads / 32) {
        if (t.r0 + r >= p.nrow) break;
        const uint8_t *row = p.src + off + (size_t)(t.r0 + r) * rowbytes;
        uint32_t w = 0;
        if (b0 + 4 <= rowbytes
            && (reinterpret_cast<uintptr_t>(row + b0) & 3u) == 0) {
            w = *reinterpret_cast<const uint32_t *>(row + b0);
        } else {
            for (int k = 0; k < 4; ++k)
                if (b0 + k < rowbytes) w |= (uint32_t)row[b0 + k] << (8 * k);
        }
        *reinterpret_cast<uint32_t *>(smem + r * kI8Pitch + 4 * lane) = w;
    }
}

// Phase 2 of decode: shared tile -> transposed float output.
template <typename OT = float>
BB_HD void i8_dec_store(const I8Geom &p, const uint8_t *smem, uint32_t block,
                        uint32_t tid) {
    I8Tile t = i8_tile(p, block);
    const long long off = p.unit_offset[t.unit];
    if (off < 0) return;
    const uint32_t tc = kI8RowBytes / p.ib;               // tile columns
    const uint32_t tr = p.nrow - t.r0 < (uint32_t)kI8Rows ? p.nrow - t.r0
                                                          : kI8Rows;
    const long long cb = p.col_begin[t.unit], ce = p.col_end[t.unit];
    const long long oc0 = p.out_col0[t.unit];
    const uint32_t total = tc * tr;
    for (uint32_t idx = tid; idx < total; idx += kI8Threads) {
        uint32_t c = tr == kI8Rows ? idx >> 5 : idx / tr;
        uint32_t r = tr == kI8Rows ? idx & 31u : idx - c * tr;
        long long j = (long long)t.j0 + c;
        if (j < cb || j >= ce || j >= (long long)p.ncol) continue;
        size_t o = (size_t)(oc0 + j - cb) * p.nrow + t.r0 + r;
        const int8_t *s = reinterpret_cast<const int8_t *>(
            smem + r * kI8Pitch + c * p.ib);
        if (p.ib == 2)
            store2(out_as<OT>(p) + 2 * o, F2{(float)s[0], (float)s[1]});
        else
            store1(out_as<OT>(p) + o, (float)s[0]);
    }
}

// Encode phase 1: float input (column-major items) -> int8 in the tile.  The
// encoders read storage type S and quantise in arith_t<S> (bb_common.cuh).
template <typename S>
BB_HD void i8_enc_load(const I8Geom &p, uint8_t *smem, uint32_t block,
                       uint32_t tid) {
    I8Tile t = i8_tile(p, block);
    if (p.unit_offset[t.unit] < 0) return;
    const uint32_t tc = kI8RowBytes / p.ib;
    const uint32_t tr = p.nrow - t.r0 < (uint32_t)kI8Rows ? p.nrow - t.r0
                                                          : kI8Rows;
    using T = arith_t<S>;
    const S *in = reinterpret_cast<const S *>(p.in);
    const uint32_t total = tc * tr;
    for (uint32_t idx = tid; idx < total; idx += kI8Threads) {
        uint32_t c = tr == kI8Rows ? idx >> 5 : idx / tr;
        uint32_t r = tr == kI8Rows ? idx & 31u : idx - c * tr;
        size_t j = (size_t)t.j0 + c;
        if (j >= p.ncol) continue;
        size_t o = ((size_t)t.unit * p.ncol + j) * p.nrow + t.r0 + r;
        uint8_t *s = smem + r * kI8Pitch + c * p.ib;
        for (uint32_t k = 0; k < p.ib; ++k)
            s[k] = (uint8_t)quant_sint<T, 8>(widen(in[o * p.ib + k]));
    }
}

// Encode phase 2: tile rows -> packed output.
BB_HD void i8_enc_store(const I8Geom &p, const uint8_t *smem, uint32_t block,
                        uint32_t tid) {
    I8Tile t = i8_tile(p, block);
    const long long off = p.unit_offset[t.unit];
    if (off < 0) return;
    const uint32_t lane = tid & 31u, warp = tid >> 5;
    const size_t rowbytes = (size_t)p.ncol * p.ib;
    const size_t b0 = (size_t)t.j0 * p.ib + 4 * lane;
    uint8_t *dst = const_cast<uint8_t *>(p.src);
    for (uint32_t r = warp; r < kI8Rows; r += kI8Threads / 32) {
        if (t.r0 + r >= p.nrow) break;
        uint8_t *row = dst + off + (size_t)(t.r0 + r) * rowbytes;
        uint32_t w = *reinterpret_cast<const uint32_t *>(
            smem + r * kI8Pitch + 4 * lane);
        if (b0 + 4 <= rowbytes
            && (reinterpret_cast<uintptr_t>(row + b0) & 3u) == 0) {
            *reinterpret_cast<uint32_t *>(row + b0) = w;
        } else {
            for (int k = 0; k < 4; ++k)
                if (b0 + k < rowbytes) row[b0 + k] = (uint8_t)(w >> (8 * k));
        }
    }
}

// ------------------------------------------------------------------------
// Fast decode path (even nrow, 16-byte aligned out): a CTA moves a tile of
// 64 rows x 256 bytes.  Shared memory is addressed in 32-bit words with an
// XOR swizzle instead of padding: word wl of row r lives at
//     r * 64 + ((wl & 32) | ((wl ^ (r >> 1)) & 31))
// so that (phase 1) a warp writing 32 consecutive words of one row and
// (phase 2) a warp reading word wc of rows 2l and 2l+1 (l = lane) both hit 32
// different banks.  In phase 2 a lane combines rows 2l and 2l+1: for complex
// items one float4 = (re, im) of two neighbouring rows, so every warp store
// instruction writes 512 contiguous bytes of one output column.  Tiles are
// ordered row-tile fastest, so neighbouring CTAs complete whole output rows.
constexpr int kF8Rows = 64;
constexpr int kF8Words = 64;               // 256 bytes per tile row
constexpr int kF8Threads = 256;
constexpr int kF8SmemWords = kF8Rows * kF8Words;

struct F8Tile { uint32_t unit, r0, w0; };  // w0: first 32-bit word in the row

// Tile order within a unit: groups of `group` column tiles x all row tiles,
// column tile fastest inside a group.  CTAs that run at the same time then
// read `group` * 256 contiguous bytes of every row (spread over the DRAM
// channels, no power-of-two row-stride camping) and together complete whole
// output rows.
BB_HD F8Tile f8_tile(const I8Geom &p, uint32_t block) {
    F8Tile t;
    const uint32_t per_unit = p.tiles_r * p.tiles_c;
    t.unit = block / per_unit;
    const uint32_t rem = block - t.unit * per_unit;
    const uint32_t per_group = p.group * p.tiles_r;
    const uint32_t g = rem / per_group;
    const uint32_t in = rem - g * per_group;
    const uint32_t left = p.tiles_c - g * p.group;
    const uint32_t width = left < p.group ? left : p.group;
    const uint32_t tr = in / width;
    t.r0 = tr * kF8Rows;
    t.w0 = (g * p.group + (in - tr * width)) * kF8Words;
    return t;
}

BB_HD uint32_t f8_swz(uint32_t r, uint32_t wl) {
    return r * kF8Words + ((wl & 32u) | ((wl ^ (r >> 1)) & 31u));
}

// Does the tile hold any column of the unit's window?
BB_HD bool f8_live(const I8Geom &p, const F8Tile &t, long long off) {
    if (off < 0) return false;
    const long long j0 = (long long)t.w0 * 4 / p.ib;
    const long long j1 = j0 + kF8Words * 4 / p.ib;
    return j0 < p.col_end[t.unit] && j1 > p.col_begin[t.unit];
}

BB_HD void f8_dec_load(const I8Geom &p, uint32_t *smem, uint32_t block,
                       uint32_t tid) {
    const F8Tile t = f8_tile(p, block);
    const long long off = p.unit_offset[t.unit];
    if (!f8_live(p, t, off)) return;
    const uint32_t lane = tid & 31u, warp = tid >> 5;
    const size_t rowbytes = (size_t)p.ncol * p.ib;
    const uint8_t *base = p.src + off;
    const bool aligned = ((reinterpret_cast<uintptr_t>(base) | rowbytes) & 3u)
        == 0;
    constexpr int kIter = kF8Rows / (kF8Threads / 32);       // 8
    if (aligned && ((size_t)t.w0 + kF8Words) * 4 <= rowbytes
        && t.r0 + kF8Rows <= p.nrow) {
        // Interior tile (CTA-uniform test): 16 unconditional loads per thread
        // are issued back to back before the first shared-memory store, so
        // 2 KiB per warp are in flight; the load phase is latency bound.
        uint32_t w[kIter][2];
        const uint8_t *col = base + (size_t)t.r0 * rowbytes
            + ((size_t)t.w0 + lane) * 4;
#pragma unroll
        for (int i = 0; i < kIter; ++i) {
            const uint8_t *q = col + (size_t)(warp + i * (kF8Threads / 32))
                * rowbytes;
            w[i][0] = *reinterpret_cast<const uint32_t *>(q);
            w[i][1] = *reinterpret_cast<const uint32_t *>(q + 128);
        }
#pragma unroll
        for (int i = 0; i < kIter; ++i) {
            const uint32_t r = warp + i * (kF8Threads / 32);
            smem[f8_swz(r, lane)] = w[i][0];
            smem[f8_swz(r, 32u + lane)] = w[i][1];
        }
        return;
    }
    // Edge tile or unaligned rows: bounds-checked, bytewise if needed.
#pragma unroll 1
    for (int i = 0; i < kIter; ++i) {
        const uint32_t r = warp + i * (kF8Threads / 32);
        if (t.r0 + r >= p.nrow) break;
        const uint8_t *row = base + (size_t)(t.r0 + r) * rowbytes;
        for (uint32_t seg = 0; seg < 2; ++seg) {
            const size_t b = ((size_t)t.w0 + seg * 32u + lane) * 4;
            uint32_t v = 0;
            if (aligned && b + 4 <= rowbytes) {
                v = *reinterpret_cast<const uint32_t *>(row + b);
            } else {
                for (int k = 0; k < 4; ++k)
                    if (b + k < rowbytes) v |= (uint32_t)row[b + k] << (8 * k);
            }
            smem[f8_swz(r, seg * 32u + lane)] = v;
        }
    }
}

BB_HD float f8_byte(uint32_t w, int k) {
    return small_int_to_float((int32_t)(int8_t)(w >> (8 * k)));
}

template <typename OT = float>
BB_HD void f8_dec_store(const I8Geom &p, const uint32_t *smem, uint32_t block,
                        uint32_t tid) {
    const F8Tile t = f8_tile(p, block);
    const long long off = p.unit_offset[t.unit];
    if (!f8_live(p, t, off)) return;
    const uint32_t lane = tid & 31u, warp = tid >> 5;
    const uint32_t ra = 2u * lane;
    if (t.r0 + ra >= p.nrow) return;                 // nrow is even
    const long long cb = p.col_begin[t.unit], ce = p.col_end[t.unit];
    const long long lim = ce < (long long)p.ncol ? ce : (long long)p.ncol;
    const long long oc0 = p.out_col0[t.unit];
    const size_t row = (size_t)t.r0 + ra;
#pragma unroll 2
    for (uint32_t wc = warp; wc < (uint32_t)kF8Words; wc += kF8Threads / 32) {
        const uint32_t a = smem[f8_swz(ra, wc)];
        const uint32_t b = smem[f8_swz(ra + 1, wc)];
        if (p.ib == 2) {
            const long long j = ((long long)t.w0 + wc) * 2;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const long long jk = j + k;
                if (jk < cb || jk >= lim) continue;
                const size_t o = (size_t)(oc0 + jk - cb) * p.nrow + row;
                store4(out_as<OT>(p) + 2 * o, F4{
                    f8_byte(a, 2 * k), f8_byte(a, 2 * k + 1),
                    f8_byte(b, 2 * k), f8_byte(b, 2 * k + 1)});
            }
        } else {
            const long long j = ((long long)t.w0 + wc) * 4;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const long long jk = j + k;
                if (jk < cb || jk >= lim) continue;
                const size_t o = (size_t)(oc0 + jk - cb) * p.nrow + row;
                store2(out_as<OT>(p) + o, F2{f8_byte(a, k), f8_byte(b, k)});
            }
        }
    }
}

// ---- fast encode: the mirror image.  Phase 1: a lane reads the (re, im) of
// rows 2l and 2l+1 of one output column as one float4 (a warp load is 512
// contiguous bytes), quantises and writes two swizzled words; phase 2: a warp
// writes 128 contiguous bytes of one packed row.
template <typename S>
BB_HD void f8_enc_load(const I8Geom &p, uint32_t *smem, uint32_t block,
                       uint32_t tid) {
    using T = arith_t<S>;
    const F8Tile t = f8_tile(p, block);
    if (p.unit_offset[t.unit] < 0) return;
    const uint32_t lane = tid & 31u, warp = tid >> 5;
    const uint32_t ra = 2u * lane;
    const bool rows_ok = t.r0 + ra < p.nrow;              // nrow is even
    const S *in = reinterpret_cast<const S *>(p.in);
    const size_t row = (size_t)t.r0 + ra;
    const size_t col0 = (size_t)t.unit * p.ncol;
    constexpr int kIter = kF8Words / (kF8Threads / 32);    // 8
    if (sizeof(T) == 4 && p.ib == 2 && t.r0 + kF8Rows <= p.nrow
        && ((size_t)t.w0 + kF8Words) * 2 <= p.ncol) {
        // Interior complex tile with float arithmetic (float32 or 16-bit
        // input; CTA-uniform test): the eight four-value loads of four word
        // columns are issued back to back before the first is quantised
        // (4 KiB per warp in flight for float32), as in the decode.
        const size_t colstride = 2 * (size_t)p.nrow;       // values per column
        constexpr int kBatch = 4;
#pragma unroll
        for (int i0 = 0; i0 < kIter; i0 += kBatch) {
            T v[kBatch][2][4];
#pragma unroll
            for (int i = 0; i < kBatch; ++i) {
                const uint32_t wc = warp + (i0 + i) * (kF8Threads / 32);
                const S *q = in
                    + 2 * ((col0 + ((size_t)t.w0 + wc) * 2) * p.nrow + row);
                load4(q, v[i][0]);
                load4(q + colstride, v[i][1]);
            }
#pragma unroll
            for (int i = 0; i < kBatch; ++i) {
                const uint32_t wc = warp + (i0 + i) * (kF8Threads / 32);
                const uint32_t a = quant_sint<T, 8>(v[i][0][0])
                    | (quant_sint<T, 8>(v[i][0][1]) << 8)
                    | (quant_sint<T, 8>(v[i][1][0]) << 16)
                    | (quant_sint<T, 8>(v[i][1][1]) << 24);
                const uint32_t b = quant_sint<T, 8>(v[i][0][2])
                    | (quant_sint<T, 8>(v[i][0][3]) << 8)
                    | (quant_sint<T, 8>(v[i][1][2]) << 16)
                    | (quant_sint<T, 8>(v[i][1][3]) << 24);
                smem[f8_swz(ra, wc)] = a;
                smem[f8_swz(ra + 1, wc)] = b;
            }
        }
        return;
    }
#pragma unroll 2
    for (int i = 0; i < kIter; ++i) {
        const uint32_t wc = warp + i * (kF8Threads / 32);
        uint32_t a = 0u, b = 0u;
        if (rows_ok) {
            if (p.ib == 2) {
                const size_t j = ((size_t)t.w0 + wc) * 2;
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    if (j + k >= p.ncol) continue;
                    T v[4];
                    load4(in + 2 * ((col0 + j + k) * p.nrow + row), v);
                    a |= (quant_sint<T, 8>(v[0])
                          | (quant_sint<T, 8>(v[1]) << 8)) << (16 * k);
                    b |= (quant_sint<T, 8>(v[2])
                          | (quant_sint<T, 8>(v[3]) << 8)) << (16 * k);
                }
            } else {
                const size_t j = ((size_t)t.w0 + wc) * 4;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (j + k >= p.ncol) continue;
                    const S *q = in + (col0 + j + k) * p.nrow + row;
                    a |= quant_sint<T, 8>(widen(q[0])) << (8 * k);
                    b |= quant_sint<T, 8>(widen(q[1])) << (8 * k);
                }
            }
        }
        smem[f8_swz(ra, wc)] = a;
        smem[f8_swz(ra + 1, wc)] = b;
    }
}

BB_HD void f8_enc_store(const I8Geom &p, const uint32_t *smem, uint32_t block,
                        uint32_t tid) {
    const F8Tile t = f8_tile(p, block);
    const long long off = p.unit_offset[t.unit];
    if (off < 0) return;
    const uint32_t lane = tid & 31u, warp = tid >> 5;
    const size_t rowbytes = (size_t)p.ncol * p.ib;
    uint8_t *base = const_cast<uint8_t *>(p.src) + off;
    const bool aligned = ((reinterpret_cast<uintptr_t>(base) | rowbytes) & 3u)
        == 0;
    constexpr int kIter = kF8Rows / (kF8Threads / 32);
#pragma unroll 2
    for (int i = 0; i < kIter; ++i) {
        const uint32_t r = warp + i * (kF8Threads / 32);
        if (t.r0 + r >= p.nrow) break;
        uint8_t *row = base + (size_t)(t.r0 + r) * rowbytes;
#pragma unroll
        for (uint32_t seg = 0; seg < 2; ++seg) {
            const uint32_t wl = seg * 32u + lane;
            const size_t b = ((size_t)t.w0 + wl) * 4;
            const uint32_t w = smem[f8_swz(r, wl)];
            if (aligned && b + 4 <= rowbytes) {
                *reinterpret_cast<uint32_t *>(row + b) = w;
            } else {
                for (int k = 0; k < 4; ++k)
                    if (b + k < rowbytes) row[b + k] = (uint8_t)(w >> (8 * k));
            }
        }
    }
}

// ------------------------------------------------------------------------
// Time-first GUPPI payloads (baseband/guppi/payload.py:97-102, :131-134):
//     in  unit: [nsample][nchan][npol] items of IB int8 (1 real, 2 complex)
//     out     : [sample][npol][nchan] items -> IB floats each
// i.e. within every time sample the (chan, pol) axes swap.  Vector path
// (nchan * IB a multiple of 4, npol 1, 2 or 4): an item is one group of
// 4 / IB channels of one sample = 4 * npol CONTIGUOUS input bytes, read with
// one 4/8/16-byte load (consecutive lanes read consecutive groups), and npol
// float4 stores, one per polarisation row; each of those warp stores covers
// 512 contiguous bytes.  Anything else: one float per item, bytewise.
struct TFGeom {
    const uint8_t *src;              // decode input / encode output
    const long long *unit_offset;    // [nunit]
    const long long *t_begin, *t_end, *out_t0;      // decode only
    void *out;                       // float32, F16 or BF16 elements
    const void *in;                  // encode input
    uint32_t nunit, nsample, nchan, npol, ib, vec;
    uint32_t sample_floats;          // npol * nchan * ib
    uint32_t row_floats;             // nchan * ib
    uint32_t items_per_unit;
    FastDiv div_sample_items, div_row_floats;
};

BB_HD uint32_t tf_get_byte(const uint32_t *w, int i) {
    return (w[i >> 2] >> (8 * (i & 3))) & 0xffu;
}

// The 4 * NPOL bytes of (sample t, channel group cg), as NPOL words.
template <int NPOL>
BB_HD void tf_load_group(const uint8_t *s, uint32_t w[NPOL]) {
    if ((reinterpret_cast<uintptr_t>(s) & (4 * NPOL - 1)) == 0) {
        if (NPOL == 4) {
            const F4 v = *reinterpret_cast<const F4 *>(s);   // 16-byte load
            const uint32_t *u = reinterpret_cast<const uint32_t *>(&v);
#pragma unroll
            for (int i = 0; i < NPOL; ++i) w[i] = u[i];
        } else if (NPOL == 2) {
            const F2 v = *reinterpret_cast<const F2 *>(s);   // 8-byte load
            const uint32_t *u = reinterpret_cast<const uint32_t *>(&v);
#pragma unroll
            for (int i = 0; i < NPOL; ++i) w[i] = u[i];
        } else {
            w[0] = *reinterpret_cast<const uint32_t *>(s);
        }
        return;
    }
#pragma unroll
    for (int i = 0; i < NPOL; ++i)
        w[i] = (uint32_t)s[4 * i] | ((uint32_t)s[4 * i + 1] << 8)
            | ((uint32_t)s[4 * i + 2] << 16) | ((uint32_t)s[4 * i + 3] << 24);
}

template <int NPOL>
BB_HD void tf_store_group(uint8_t *d, const uint32_t w[NPOL]) {
    if ((reinterpret_cast<uintptr_t>(d) & (4 * NPOL - 1)) == 0) {
        if (NPOL == 4) {
            F4 v;
            uint32_t *u = reinterpret_cast<uint32_t *>(&v);
#pragma unroll
            for (int i = 0; i < NPOL; ++i) u[i] = w[i];
            *reinterpret_cast<F4 *>(d) = v;
        } else if (NPOL == 2) {
            F2 v;
            uint32_t *u = reinterpret_cast<uint32_t *>(&v);
#pragma unroll
            for (int i = 0; i < NPOL; ++i) u[i] = w[i];
            *reinterpret_cast<F2 *>(d) = v;
        } else {
            *reinterpret_cast<uint32_t *>(d) = w[0];
        }
        return;
    }
#pragma unroll
    for (int i = 0; i < 4 * NPOL; ++i) d[i] = (uint8_t)tf_get_byte(w, i);
}

BB_HD float tf_f(uint32_t b) {
    return small_int_to_float((int32_t)(int8_t)b);
}

template <int NPOL, typename OT>
BB_HD void tf_decode_group(const TFGeom &p, uint32_t unit, uint32_t item,
                           long long off) {
    uint32_t t_rel, cg;
    p.div_sample_items.divmod(item, t_rel, cg);
    const long long t = p.t_begin[unit] + t_rel;
    if (t >= p.t_end[unit] || t >= (long long)p.nsample) return;
    uint32_t w[NPOL];
    tf_load_group<NPOL>(p.src + off
                        + ((size_t)t * (p.row_floats / 4) + cg) * (4 * NPOL), w);
    OT *dst = out_as<OT>(p) + ((size_t)(p.out_t0[unit] + t_rel)
                               * p.sample_floats + 4 * cg);
#pragma unroll
    for (int pol = 0; pol < NPOL; ++pol) {
        F4 v;
        if (p.ib == 2) {             // bytes [chan 0..1][pol][re, im]
            const int i0 = 2 * pol, i1 = 2 * (NPOL + pol);
            v = F4{tf_f(tf_get_byte(w, i0)), tf_f(tf_get_byte(w, i0 + 1)),
                   tf_f(tf_get_byte(w, i1)), tf_f(tf_get_byte(w, i1 + 1))};
        } else {                     // bytes [chan 0..3][pol]
            v = F4{tf_f(tf_get_byte(w, pol)), tf_f(tf_get_byte(w, NPOL + pol)),
                   tf_f(tf_get_byte(w, 2 * NPOL + pol)),
                   tf_f(tf_get_byte(w, 3 * NPOL + pol))};
        }
        store4(dst + (size_t)pol * p.row_floats, v);
    }
}

template <typename OT = float>
BB_HD void tf_decode(const TFGeom &p, uint32_t unit, uint32_t item) {
    if (item >= p.items_per_unit) return;
    const long long off = p.unit_offset[unit];
    if (off < 0) return;
    if (p.vec == 4) {
        if (p.npol == 2) tf_decode_group<2, OT>(p, unit, item, off);
        else if (p.npol == 4) tf_decode_group<4, OT>(p, unit, item, off);
        else tf_decode_group<1, OT>(p, unit, item, off);
        return;
    }
    // one float per item: (sample, pol, chan, component)
    uint32_t t_rel, r, pol, f;
    p.div_sample_items.divmod(item, t_rel, r);
    p.div_row_floats.divmod(r, pol, f);
    const long long t = p.t_begin[unit] + t_rel;
    if (t >= p.t_end[unit] || t >= (long long)p.nsample) return;
    const uint32_t chan = p.ib == 2 ? f >> 1 : f, k = p.ib == 2 ? (f & 1u) : 0u;
    const int8_t *s = reinterpret_cast<const int8_t *>(p.src + off);
    store1(out_as<OT>(p) + (size_t)(p.out_t0[unit] + t_rel) * p.sample_floats
           + r,
           (float)s[(((size_t)t * p.nchan + chan) * p.npol + pol) * p.ib + k]);
}

template <typename S, int NPOL>
BB_HD void tf_encode_group(const TFGeom &p, uint32_t unit, uint32_t item,
                           long long off) {
    using T = arith_t<S>;
    uint32_t t, cg;
    p.div_sample_items.divmod(item, t, cg);
    const S *q = reinterpret_cast<const S *>(p.in)
        + (((size_t)unit * p.nsample + t) * p.sample_floats + 4 * cg);
    T v[NPOL][4];
#pragma unroll
    for (int pol = 0; pol < NPOL; ++pol)
        load4(q + (size_t)pol * p.row_floats, v[pol]);
    uint32_t w[NPOL];
#pragma unroll
    for (int i = 0; i < NPOL; ++i) w[i] = 0u;
#pragma unroll
    for (int pol = 0; pol < NPOL; ++pol) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            // float j of the row piece -> byte position within the group
            const int i2 = 2 * ((j >> 1) * NPOL + pol) + (j & 1);
            const int i1 = j * NPOL + pol;
            const uint32_t code = quant_sint<T, 8>(v[pol][j]);
            if (p.ib == 2) w[i2 >> 2] |= code << (8 * (i2 & 3));
            else w[i1 >> 2] |= code << (8 * (i1 & 3));
        }
    }
    tf_store_group<NPOL>(const_cast<uint8_t *>(p.src) + off
                         + ((size_t)t * (p.row_floats / 4) + cg) * (4 * NPOL),
                         w);
}

template <typename S>
BB_HD void tf_encode(const TFGeom &p, uint32_t unit, uint32_t item) {
    if (item >= p.items_per_unit) return;
    const long long off = p.unit_offset[unit];
    if (off < 0) return;
    if (p.vec == 4) {
        if (p.npol == 2) tf_encode_group<S, 2>(p, unit, item, off);
        else if (p.npol == 4) tf_encode_group<S, 4>(p, unit, item, off);
        else tf_encode_group<S, 1>(p, unit, item, off);
        return;
    }
    uint32_t t, r, pol, f;
    p.div_sample_items.divmod(item, t, r);
    p.div_row_floats.divmod(r, pol, f);
    const uint32_t chan = p.ib == 2 ? f >> 1 : f, k = p.ib == 2 ? (f & 1u) : 0u;
    const S *q = reinterpret_cast<const S *>(p.in)
        + (((size_t)unit * p.nsample + t) * p.sample_floats + r);
    const_cast<uint8_t *>(p.src)[off + (((size_t)t * p.nchan + chan) * p.npol
                                        + pol) * p.ib + k] =
        (uint8_t)quant_sint<arith_t<S>, 8>(widen(q[0]));
}

// Host-side validation / geometry shared with the CPU emulation.
inline const char *tf_fill_geom(TFGeom &g, int64_t nunit, int64_t nsample,
                                int32_t nchan, int32_t npol,
                                int32_t item_nbytes, bool aligned16) {
    if (item_nbytes != 1 && item_nbytes != 2)
        return "item_nbytes must be 1 or 2";
    if (nunit < 0 || nunit > 65535 || nsample < 1 || nchan < 1 || npol < 1)
        return "bad nunit/nsample/nchan/npol";
    const uint64_t rf = (uint64_t)nchan * item_nbytes;
    const uint64_t sf = rf * npol;
    const bool vec = aligned16 && rf % 4 == 0
        && (npol == 1 || npol == 2 || npol == 4);
    // items per sample: channel groups (vector path) or floats
    const uint64_t per_sample = vec ? rf / 4 : sf;
    const uint64_t items = (uint64_t)nsample * per_sample;
    if (sf > 0x7fffffffull || items > 0xffffffffull)
        return "unit too large for one call; split it along time";
    g.nunit = (uint32_t)nunit;
    g.nsample = (uint32_t)nsample;
    g.nchan = (uint32_t)nchan;
    g.npol = (uint32_t)npol;
    g.ib = (uint32_t)item_nbytes;
    g.vec = vec ? 4 : 1;
    g.sample_floats = (uint32_t)sf;
    g.row_floats = (uint32_t)rf;
    g.items_per_unit = (uint32_t)items;
    g.div_sample_items = make_fastdiv((uint32_t)per_sample);
    g.div_row_floats = make_fastdiv((uint32_t)rf);
    return nullptr;
}

}  // namespace bb
