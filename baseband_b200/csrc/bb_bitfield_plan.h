// Host-side planning for the bit-field codec: validates a call, picks the
// work decomposition and splits it into launches whose item counts fit in 32
// bits.  Pure C++ so the CPU emulation in tests/emu shares it.
#pragma once
#include <stdlib.h>
#include <vector>
#include <string>
#include "bb_bitfield.cuh"

namespace bb {

enum { MODE_ROWGROUP4 = 0, MODE_ROWGROUP2 = 1, MODE_RUN = 2, MODE_SCALAR = 3,
       MODE_WORDRUN = 4, MODE_WORDROW4 = 7, MODE_ROWWORD4 = 8,
       MODE_ROWWORD2 = 9, MODE_WORDROW2 = 10,
       MODE_WORDROW4X2 = 11, MODE_WORDROW2X2 = 12,     // rows of two float4
       MODE_TILE4 = 13, MODE_TILE2 = 14,               // rows of four float4
       MODE_RUNS = 15,          // RUN, one word -> its S samples as S rows
       MODE_RUNQ = 16 };        // 8-bit encode: four words per item

// Development tunables (BB_TUNE_<NAME> environment variables), read at every
// call so that a sweep can change them inside one process.
inline int tune(const char *name, int dflt) {
    const char *e = getenv(name);
    return (e && *e) ? atoi(e) : dflt;
}

inline bool is_wordrow(int mode) {
    return mode == MODE_WORDROW4 || mode == MODE_WORDROW2
        || mode == MODE_WORDROW4X2 || mode == MODE_WORDROW2X2;
}

// sel: levels by register select instead of the shared-memory pair table;
// tile_p / tile_u: word positions per chunk and chunks per warp (TILE modes).
struct DecLaunch { int mode; DecGeom g; int sel = 0, tile_p = 8, tile_u = 1; };

inline bool is_tile(int mode) {
    return mode == MODE_TILE4 || mode == MODE_TILE2;
}
struct EncLaunch { int mode; EncGeom g; };   // MODE_RUN = vectorised words

inline bool plan_geometry(int64_t payload_nbytes, int bps, int nelem,
                          int nthread, int64_t nset, uint32_t &nword,
                          uint32_t &spf, std::string &err) {
    if (!(bps == 1 || bps == 2 || bps == 4 || bps == 8)) {
        err = "bps must be 1, 2, 4 or 8";
        return false;
    }
    if (nelem < 1 || nthread < 1 || nset < 0 || payload_nbytes <= 0) {
        err = "nelem, nthread >= 1, nset >= 0, payload_nbytes > 0 required";
        return false;
    }
    if (payload_nbytes % 4) {
        err = "payload_nbytes must be a multiple of 4";
        return false;
    }
    int64_t bits = payload_nbytes * 8;
    if (bits % ((int64_t)bps * nelem)) {
        err = "payload does not hold a whole number of complete samples";
        return false;
    }
    int64_t s = bits / ((int64_t)bps * nelem);
    if (payload_nbytes / 4 > 0x3fffffff || s > 0x7fffffff) {
        err = "payload too large for one unit; split it along time";
        return false;
    }
    nword = (uint32_t)(payload_nbytes / 4);
    spf = (uint32_t)s;
    return true;
}

inline int pick_mode(int nelem, int nthread, bool aligned_rows,
                     bool decode = false) {
    if (decode && nthread == 4 && nelem == 1) return MODE_WORDROW4;
    if (decode && nthread == 2 && nelem == 2) return MODE_WORDROW2;
    if (decode && nthread == 8 && nelem == 1) return MODE_WORDROW4X2;
    if (decode && nthread == 4 && nelem == 2) return MODE_WORDROW2X2;
    if (nthread > 1 && nelem == 1 && nthread % 4 == 0) return MODE_ROWGROUP4;
    if (nthread > 1 && nelem == 2 && nthread % 2 == 0) return MODE_ROWGROUP2;
    if (aligned_rows && nthread == 1) return MODE_WORDRUN;
    if (aligned_rows && nelem % 4 == 0 && ilog2_exact(nelem) >= 0)
        return MODE_RUN;
    return MODE_SCALAR;
}

inline bool plan_decode(const void *src, const int64_t *unit_offset,
                        int64_t nset, int nthread, int64_t payload_nbytes,
                        int bps, int nelem, int complex_data, float fill,
                        int64_t sample_start, int64_t nsample, void *out,
                        std::vector<DecLaunch> &launches, std::string &err) {
    uint32_t nword, spf;
    if (!plan_geometry(payload_nbytes, bps, nelem, nthread, nset, nword, spf,
                       err))
        return false;
    if (sample_start < 0 || nsample < 0
        || sample_start + nsample > nset * (int64_t)spf) {
        err = "sample range outside the given frames";
        return false;
    }
    if (nsample == 0) return true;
    const int64_t rowlen = (int64_t)nthread * nelem;
    const bool aligned_rows = (sample_start * rowlen) % 4 == 0
        && (nsample * rowlen) % 4 == 0;
    int mode = pick_mode(nelem, nthread, aligned_rows, true);
    // rows of four float4 (the C2 shape): BB_TUNE_C2 = 0 ROWGROUP + table,
    // 1 ROWGROUP + select, 2/3 TILE (8 positions) table/select, 4/5 TILE (4)
    // Per-mode default (profiles/r2_sweep_variants.txt): four real threads
    // per float4 (ROWGROUP4) select the levels in registers -- 32 registers,
    // 8 CTAs per SM, no shared-memory lookups; same burst rate as the table
    // but it holds it in long runs (6.75 vs 6.57 TB/s sustained); the complex
    // pairs of ROWGROUP2 stay with the pair table (6.78 vs 6.74).
    const int c2 = tune("BB_TUNE_C2", mode == MODE_ROWGROUP4 ? 1 : 0);
    int sel = 0, tile_p = 8;
    const int tile_u = tune("BB_TUNE_TILE_U", 1) >= 2 ? 2 : 1;
    if (bps == 2 && (mode == MODE_ROWGROUP4 || mode == MODE_ROWGROUP2)) {
        sel = c2 & 1;
        const bool row16 = (mode == MODE_ROWGROUP4 && nthread == 16)
            || (mode == MODE_ROWGROUP2 && nthread == 8);
        if (c2 >= 2 && row16) {
            mode = mode == MODE_ROWGROUP4 ? MODE_TILE4 : MODE_TILE2;
            tile_p = c2 >= 4 ? 4 : 8;
        }
    }
    const int cpw = 32 / bps;
    // several threads of several channels, S = cpw / nelem >= 1 samples per
    // word: one item per float4 position and group of R = max(S, 4) rows
    // (R / S words), if the read is aligned to R rows (else to S, S >= 2)
    const int runs_s = (mode == MODE_RUN && nthread > 1 && nelem >= 4
                        && cpw / nelem >= 1 && tune("BB_TUNE_RUNS", 1))
        ? cpw / nelem : 0;
    int runs_rows = 0;
    if (runs_s) {
        const int wide = runs_s > 4 ? runs_s : 4;
        if (sample_start % wide == 0 && nsample % wide == 0
            && spf % wide == 0)
            runs_rows = wide;
        else if (runs_s >= 2 && sample_start % runs_s == 0
                 && nsample % runs_s == 0)
            runs_rows = runs_s;
    }
    if (runs_rows) mode = MODE_RUNS;
    int64_t first = sample_start / spf;
    int64_t last = (sample_start + nsample + spf - 1) / spf;
    // items per set and the 32-bit budget for one launch
    uint64_t per_set;
    uint32_t ngroup = 1;
    if (mode == MODE_ROWGROUP4 || mode == MODE_ROWGROUP2) {
        ngroup = nthread / (mode == MODE_ROWGROUP4 ? 4 : 2);
        // words with more than 8 rows are split over several items
        const int tpw = cpw / (mode == MODE_ROWGROUP4 ? 1 : 2);
        per_set = (uint64_t)nword * ngroup * (tpw > 8 ? tpw / 8 : 1);
    } else if (mode == MODE_RUN) {
        per_set = (uint64_t)spf * rowlen / 4;
    } else if (mode == MODE_RUNS) {
        per_set = (uint64_t)spf / runs_rows * rowlen / 4;
    } else if (mode == MODE_WORDRUN || is_wordrow(mode) || is_tile(mode)) {
        per_set = nword;                  // items are lanes = words
    } else {
        per_set = (uint64_t)spf * rowlen;
    }
    const uint64_t budget = (mode == MODE_RUN || mode == MODE_RUNS)
        ? 0x3fffffffull
        : (mode == MODE_WORDRUN || is_wordrow(mode) || is_tile(mode))
        ? 0x03ffffffull : 0x7fffffffull;
    if (per_set > budget) {
        err = "one frame set is too large for a launch; split it along time";
        return false;
    }
    int64_t max_sets = (int64_t)(budget / per_set);
    for (int64_t s0 = first; s0 < last; s0 += max_sets) {
        int64_t s1 = s0 + max_sets < last ? s0 + max_sets : last;
        DecGeom g;
        g.src = (const uint8_t *)src;
        g.unit_offset = (const long long *)unit_offset + s0 * nthread;
        g.out = out;
        g.row_base = s0 * (int64_t)spf - sample_start;
        g.nsample = nsample;
        g.nset = (uint32_t)(s1 - s0);
        g.nthread = nthread;
        g.nelem = nelem;
        g.nword = nword;
        g.tpw = cpw / nelem ? cpw / nelem : 1;
        g.spf = spf;
        g.nitems = (uint32_t)(per_set * (uint64_t)(s1 - s0));
        g.nwords_total = (uint32_t)((uint64_t)nword * (uint64_t)(s1 - s0));
        if (mode == MODE_WORDRUN || is_wordrow(mode))        // whole warps
            g.nitems = (g.nwords_total + 31u) / 32u * 32u;
        if (is_tile(mode))                // a warp per tile_p word positions
            g.nitems = (g.nwords_total + tile_p - 1u) / tile_p * 32u;
        g.ngroup = ngroup;
        g.log2_nelem = ilog2_exact(nelem);
        g.complex_fill = complex_data ? 1 : 0;
        g.debug = (uint32_t)tune("BB_TUNE_KNOCK", 0);
        g.fill = fill;
        g.div_nword = make_fastdiv(nword);
        g.div_ngroup = make_fastdiv(ngroup);
        g.div_rowlen = make_fastdiv((uint32_t)rowlen);
        g.div_spf = make_fastdiv(spf);
        g.div_nelem = make_fastdiv(nelem);
        g.div_unitlen = make_fastdiv((uint32_t)((uint64_t)spf * nelem));
        g.div_f4row = make_fastdiv((uint32_t)(rowlen / 4 ? rowlen / 4 : 1));
        g.runs_rows = (uint32_t)runs_rows;
        DecLaunch l;
        l.mode = mode;
        l.g = g;
        l.sel = sel;
        l.tile_p = tile_p;
        l.tile_u = tile_u;
        launches.push_back(l);
    }
    return true;
}

inline bool plan_encode(const void *in, void *dst, const int64_t *unit_offset,
                        int64_t nset, int nthread, int64_t payload_nbytes,
                        int bps, int nelem, std::vector<EncLaunch> &launches,
                        std::string &err) {
    uint32_t nword, spf;
    if (!plan_geometry(payload_nbytes, bps, nelem, nthread, nset, nword, spf,
                       err))
        return false;
    if (nset == 0) return true;
    const int64_t rowlen = (int64_t)nthread * nelem;
    int mode = pick_mode(nelem, nthread, true);
    if (mode == MODE_WORDRUN) mode = MODE_RUN;   // encode: vectorised words
    // a row is one float4: warp-cooperative rows -> words
    const uint64_t rw_budget = 0x03ffffffull;    // word positions per launch
    // (measured: it wins from 8 rows per word on; below that ROWGROUP's
    // 32/64-byte pieces per lane coalesce well enough)
    if (mode == MODE_ROWGROUP4 && nthread == 4 && nword <= rw_budget
        && bps <= 4)
        mode = MODE_ROWWORD4;
    if (mode == MODE_ROWGROUP2 && nthread == 2 && nword <= rw_budget
        && bps <= 2)
        mode = MODE_ROWWORD2;
    // 8 bit, whole words of one row segment in fours (one thread, or >= 16
    // elements per thread row): an item is four words -- the divisions and
    // the unit-offset load once per 64 input bytes, one 16-byte store
    if (mode == MODE_RUN && bps == 8 && nword % 4 == 0
        && (nthread == 1 || nelem % 16 == 0) && tune("BB_TUNE_RUNQ", 1))
        mode = MODE_RUNQ;
    uint64_t per_set;
    uint32_t ngroup = 1;
    if (mode == MODE_ROWGROUP4 || mode == MODE_ROWGROUP2) {
        ngroup = nthread / (mode == MODE_ROWGROUP4 ? 4 : 2);
        per_set = (uint64_t)nword * ngroup;
    } else if (mode == MODE_ROWWORD4 || mode == MODE_ROWWORD2) {
        per_set = nword;                  // items are lanes = word positions
    } else if (mode == MODE_RUNQ) {
        per_set = (uint64_t)(nword / 4) * nthread;
    } else {
        per_set = (uint64_t)nword * nthread;
    }
    if (per_set > 0x7fffffffull) {
        err = "one frame set is too large for a launch; split it along time";
        return false;
    }
    int64_t max_sets = (int64_t)(((mode == MODE_ROWWORD4
                                   || mode == MODE_ROWWORD2) ? rw_budget
                                  : 0x7fffffffull) / per_set);
    for (int64_t s0 = 0; s0 < nset; s0 += max_sets) {
        int64_t s1 = s0 + max_sets < nset ? s0 + max_sets : nset;
        EncGeom g;
        g.in = in;
        g.in_elem_offset = (unsigned long long)(s0 * (int64_t)spf * rowlen);
        g.dst = (uint8_t *)dst;
        g.unit_offset = (const long long *)unit_offset + s0 * nthread;
        g.nset = (uint32_t)(s1 - s0);
        g.nthread = nthread;
        g.nelem = nelem;
        g.nword = nword;
        g.spf = spf;
        g.nitems = (uint32_t)(per_set * (uint64_t)(s1 - s0));
        g.nwords_total = (uint32_t)((uint64_t)nword * (uint64_t)(s1 - s0));
        if (mode == MODE_ROWWORD4 || mode == MODE_ROWWORD2)   // whole warps
            g.nitems = (g.nwords_total + 31u) / 32u * 32u;
        g.ngroup = ngroup;
        g.log2_nelem = ilog2_exact(nelem);
        g.div_nword = make_fastdiv(mode == MODE_RUNQ ? nword / 4 : nword);
        g.div_ngroup = make_fastdiv(ngroup);
        g.div_nthread = make_fastdiv(nthread);
        launches.push_back({mode, g});
    }
    return true;
}

}  // namespace bb
