// Selective decoders: per-thread bodies and host planning.
//
// Only the selected components of every decoded row are written:
//     out[row * nsel + j] = full_row[sel[j]]
// in float32, F16 or BF16, so a `subset` read costs what it selects.  Two
// layouts, one body:
//   BITFIELD  the units of bb_decode_bitfield; sel[j] is a component index
//             slot * nelem + e of the decoded row (nthread * nelem wide), and
//             component (slot, e) of row (set, t) is the code at bit
//             (t * nelem + e) * bps of unit (set, slot).  Invalid units
//             (offset < 0) give fill_value, 0 for imaginary components of
//             complex data, as bb_decode_bitfield writes.
//   INT8      int8 units with an axis transpose (GUPPI channels-first and
//             time-first, MKBF heaps); sel[j] is the byte offset of component
//             j at time 0 of a unit, and time t sits
//             (t / heap) * heap_stride + (t % heap) * t_stride further on.
//             Unit u contributes samples [t_begin[u], t_end[u]) to the output
//             rows from out_t0[u] on (the window tables of the int8 decoders).
//
// Decomposition by output position: a thread owns kSelGroups groups of four
// consecutive output elements, aligned to 4-element boundaries of the output
// address (16 bytes of float32, 8 of the 16-bit types) and kSelThreads apart,
// so every warp store covers contiguous bytes (512 for float32) whatever nsel
// is, and any output alignment and any nsel work: groups cut by the ends of
// the range store element by element.  All loads of a thread are issued
// before its first decode; neighbouring outputs read neighbouring (often the
// same) packed words, which L1 serves.  The table is resolved once per CTA
// into shared memory when it is at most kSelSmem entries, else read per
// element (it is then as large as the CTA's share of the output).
#pragma once
#include <string>
#include <vector>
#include "bb_bitfield_plan.h"

namespace bb {

constexpr int kSelThreads = 256;
constexpr int kSelGroups = 4;            // float4 groups per thread
constexpr uint32_t kSelSmem = 2048;      // table entries kept in shared memory

// One table entry: BITFIELD (slot, e), INT8 (0, byte offset); slot < 0 marks
// an entry outside the row (written as NaN, nothing is read for it).
struct SelEntry { int32_t slot, off; };

struct SelGeom {
    const uint8_t *src;
    const long long *unit_offset;   // BITFIELD: set 0 of this launch
    const int32_t *sel;             // [nsel]
    void *out;                      // element 0 of the whole output
    uint32_t head;                  // (out address / element size) % 4
    uint32_t nsel;
    FastDiv div_nsel;
    // BITFIELD: output elements [e0, e1) of this launch, groups from g0
    long long e0, e1, g0;
    uint32_t ngroups;
    uint32_t nthread, nelem, ncomp, t_base, complex_fill, cpw_log2;
    float fill;
    FastDiv div_spf, div_nelem;
    // INT8
    const long long *t_begin, *t_end, *out_t0;
    long long heap_stride;
    long long t_stride;
    FastDiv div_heap;
};

// value kinds of an element (bits 5-6 of its meta word); bit 7: written
enum { SEL_DECODE = 0, SEL_FILL = 1, SEL_ZERO = 2, SEL_NAN = 3 };
constexpr uint32_t kSelLive = 1u << 7;

template <bool INT8>
BB_HD SelEntry sel_entry(const SelGeom &p, uint32_t j) {
    const int32_t c = p.sel[j];
    if (INT8) return SelEntry{c < 0 ? -1 : 0, c};
    if (c < 0 || (uint32_t)c >= p.ncomp) return SelEntry{-1, 0};
    uint32_t slot, e;
    p.div_nelem.divmod((uint32_t)c, slot, e);
    return SelEntry{(int32_t)slot, (int32_t)e};
}

BB_HD SelEntry sel_lookup(const SelGeom &p, const SelEntry *tab, uint32_t j,
                          bool int8) {
    if (p.nsel <= kSelSmem) return tab[j];
    return int8 ? sel_entry<true>(p, j) : sel_entry<false>(p, j);
}

// The four elements of group g (absolute: elements 4g - head .. 4g + 3 -
// head of `out`): their packed words and meta words (code position in the
// word, value kind, written).  BITFIELD: `unit` is unused; INT8: the unit and
// its output element range [ue0, ue1) (a window of rows).
template <int BPS, bool INT8>
BB_HD void sel_fetch(const SelGeom &p, const SelEntry *tab, long long g,
                     uint32_t unit, long long ue0, long long ue1,
                     uint32_t w[4], uint32_t meta[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        w[i] = 0u;
        meta[i] = 0u;
        const long long E = 4 * g + i - (long long)p.head;
        const long long lo = INT8 ? ue0 : p.e0, hi = INT8 ? ue1 : p.e1;
        if (E < lo || E >= hi) continue;
        uint32_t row, j;
        p.div_nsel.divmod((uint32_t)(E - lo), row, j);
        const SelEntry s = sel_lookup(p, tab, j, INT8);
        if (s.slot < 0) {
            meta[i] = kSelLive | (SEL_NAN << 5);
            continue;
        }
        if (INT8) {
            const long long t = p.t_begin[unit] + row;
            const long long uo = p.unit_offset[unit];
            uint32_t h, tt;
            p.div_heap.divmod((uint32_t)t, h, tt);
            w[i] = p.src[uo + h * p.heap_stride + tt * p.t_stride + s.off];
            meta[i] = kSelLive;
            continue;
        }
        uint32_t set, t;
        p.div_spf.divmod(p.t_base + row, set, t);
        const long long uo = p.unit_offset[(size_t)set * p.nthread + s.slot];
        if (uo < 0) {
            meta[i] = kSelLive | ((p.complex_fill && (s.off & 1))
                                  ? SEL_ZERO : SEL_FILL) << 5;
            continue;
        }
        const unsigned long long code =
            (unsigned long long)t * p.nelem + (uint32_t)s.off;
        w[i] = load_u32(p.src + uo + 4ull * (code >> p.cpw_log2));
        meta[i] = kSelLive | (uint32_t)(code & ((1u << p.cpw_log2) - 1u));
    }
}

template <int BPS, int CODEC>
BB_HD float sel_value(const SelGeom &p, const float *lut, uint32_t w,
                      uint32_t meta) {
    switch ((meta >> 5) & 3u) {
    case SEL_DECODE: return decode_one<BPS, CODEC>(w, meta & 31u, lut);
    case SEL_FILL: return p.fill;
    case SEL_ZERO: return 0.f;
    default: return uint_as_float(0x7fc00000u);
    }
}

template <int BPS, int CODEC, typename OT>
BB_HD void sel_emit(const SelGeom &p, const float *lut, long long g,
                    const uint32_t w[4], const uint32_t meta[4]) {
    OT *dst = out_as<OT>(p) + (4 * g - (long long)p.head);
    if (meta[0] & meta[1] & meta[2] & meta[3] & kSelLive) {
        store4(dst, F4{sel_value<BPS, CODEC>(p, lut, w[0], meta[0]),
                       sel_value<BPS, CODEC>(p, lut, w[1], meta[1]),
                       sel_value<BPS, CODEC>(p, lut, w[2], meta[2]),
                       sel_value<BPS, CODEC>(p, lut, w[3], meta[3])});
        return;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (meta[i] & kSelLive)
            store1(dst + i, sel_value<BPS, CODEC>(p, lut, w[i], meta[i]));
}

// Output element range of INT8 unit u.
BB_HD void sel_unit_range(const SelGeom &p, uint32_t u, long long &ue0,
                          long long &ue1) {
    ue0 = p.out_t0[u] * (long long)p.nsel;
    const long long n = p.t_end[u] - p.t_begin[u];
    ue1 = ue0 + (n > 0 ? n : 0) * (long long)p.nsel;
}

BB_HD long long floor4(long long x) { return x >= 0 ? x / 4 : -((3 - x) / 4); }

// ------------------------------------------------------------------ planning
inline uint32_t out_head(const void *out, int esize) {
    return (uint32_t)(((uintptr_t)out / (uintptr_t)esize) % 4u);
}

// BITFIELD: one launch per block of rows whose element and time indices fit
// in 32 bits.
inline bool plan_select_bitfield(
    const void *src, const int64_t *unit_offset, int64_t nset, int nthread,
    int64_t payload_nbytes, int bps, int nelem, int complex_data, float fill,
    int64_t sample_start, int64_t nsample, const int32_t *sel, int nsel,
    void *out, int esize, std::vector<SelGeom> &launches, std::string &err) {
    uint32_t nword, spf;
    if (!plan_geometry(payload_nbytes, bps, nelem, nthread, nset, nword, spf,
                       err))
        return false;
    if (nsel < 1) {
        err = "nsel must be at least 1";
        return false;
    }
    if ((int64_t)nthread * nelem > 0x7fffffff) {
        err = "rows too wide";
        return false;
    }
    if (sample_start < 0 || nsample < 0
        || sample_start + nsample > nset * (int64_t)spf) {
        err = "sample range outside the given frames";
        return false;
    }
    const int64_t rows_max = (0x7fffffffLL / nsel) < (0x7fffffffLL - spf)
        ? 0x7fffffffLL / nsel : 0x7fffffffLL - spf;
    const uint32_t head = out_head(out, esize);
    for (int64_t r0 = 0; r0 < nsample; r0 += rows_max) {
        const int64_t r1 = r0 + rows_max < nsample ? r0 + rows_max : nsample;
        const int64_t s = sample_start + r0;
        SelGeom g = SelGeom();
        g.src = (const uint8_t *)src;
        g.unit_offset = (const long long *)unit_offset + (s / spf) * nthread;
        g.sel = sel;
        g.out = out;
        g.head = head;
        g.nsel = (uint32_t)nsel;
        g.div_nsel = make_fastdiv((uint32_t)nsel);
        g.e0 = r0 * nsel;
        g.e1 = r1 * nsel;
        g.g0 = floor4(g.e0 + head);
        g.ngroups = (uint32_t)(floor4(g.e1 + head + 3) - g.g0);
        g.nthread = (uint32_t)nthread;
        g.nelem = (uint32_t)nelem;
        g.ncomp = (uint32_t)(nthread * nelem);
        g.t_base = (uint32_t)(s % spf);
        g.complex_fill = complex_data ? 1u : 0u;
        g.cpw_log2 = (uint32_t)ilog2_exact(32 / bps);
        g.fill = fill;
        g.div_spf = make_fastdiv(spf);
        g.div_nelem = make_fastdiv((uint32_t)nelem);
        g.div_heap = make_fastdiv(1);
        launches.push_back(g);
    }
    return true;
}

// INT8: one geometry; the caller launches (groups of the widest unit) x
// units.  Returns the number of groups a unit can have.
inline bool plan_select_int8(
    const void *src, const int64_t *unit_offset, int64_t nunit, int64_t nsample,
    int64_t heap, int64_t heap_stride, int64_t t_stride, const int32_t *off,
    int nsel, const int64_t *t_begin, const int64_t *t_end,
    const int64_t *out_t0, void *out, int esize, SelGeom &g,
    uint32_t &ngroups_max, std::string &err) {
    if (nsel < 1 || nunit < 0 || nsample < 0 || heap < 1 || heap_stride < 0
        || t_stride < 0) {
        err = "nsel, heap >= 1 and nunit, nsample, strides >= 0 required";
        return false;
    }
    if (nsample > 0xffffffffLL || heap > 0xffffffffLL
        || nsample * nsel > 0x7ffffffcLL) {
        err = "units too large for one call; split them along time";
        return false;
    }
    g = SelGeom();
    g.src = (const uint8_t *)src;
    g.unit_offset = (const long long *)unit_offset;
    g.sel = off;
    g.out = out;
    g.head = out_head(out, esize);
    g.nsel = (uint32_t)nsel;
    g.div_nsel = make_fastdiv((uint32_t)nsel);
    g.t_begin = (const long long *)t_begin;
    g.t_end = (const long long *)t_end;
    g.out_t0 = (const long long *)out_t0;
    g.heap_stride = heap_stride;
    g.t_stride = t_stride;
    g.div_heap = make_fastdiv((uint32_t)heap);
    g.div_spf = g.div_nelem = make_fastdiv(1);
    ngroups_max = (uint32_t)((nsample * nsel + 3) / 4 + 1);
    return true;
}

}  // namespace bb
