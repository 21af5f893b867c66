// Host-side planning for the Mark 4 codec (shared with the CPU emulation).
#pragma once
#include <stdlib.h>
#include <string>
#include <vector>
#include "bb_mark4.cuh"

namespace bb {

enum { M4_FAST = 0, M4_GENERIC_VEC = 1, M4_GENERIC_SCALAR = 2, M4_WARP = 3,
       M4_HALF = 4 };

struct M4Launch { int mode; M4Geom g; };

// Where input bit b of a 32-bit group ends up after reorder32
// (baseband/mark4/payload.py:48-52).
inline int m4_reorder_bit(int b) {
    if ((0xAA55AA55u >> b) & 1u) return b;
    if ((0x55005500u >> b) & 1u) return b - 7;
    return b + 7;
}

// Bit positions of (sign, magnitude) for sample f of the word and channel c,
// derived from the reference decoders (baseband/mark4/payload.py:122-288).
inline bool m4_build_pos(int nchan, int fanout, int ft, uint16_t pos[32],
                         int &ntrack, std::string &err) {
    static const int perm[4] = {0, 2, 1, 3};
    ntrack = nchan * 2 * fanout;
    const bool known = (!ft && ((nchan == 2 && fanout == 4)
                                || (nchan == 4 && fanout == 4)
                                || (nchan == 8 && fanout == 2)
                                || (nchan == 8 && fanout == 4)))
        || (ft && nchan == 16 && fanout == 2);
    if (!known) {
        err = "no Mark 4 codec for this (nchan, fanout, ft)";
        return false;
    }
    int spos[32], mpos[32];
    for (int i = 0; i < 32; ++i) spos[i] = mpos[i] = -1;
    for (int b = 0; b < ntrack; ++b) {
        int t, c, mag;
        if (nchan == 2) {                       // 16 tracks, lut2bit3
            int B = b >> 3, j = b & 7;
            c = B; t = j & 3; mag = (j >> 2) & 1;
        } else if (fanout == 4) {               // 32/64 tracks, reorder + lut2bit1
            int bp = m4_reorder_bit(b & 31);
            int byte_ = bp >> 3, j = bp & 7;
            t = j >> 1; mag = j & 1;
            c = perm[byte_] + 4 * (b >> 5);
        } else if (!ft) {                       // 32 tracks, 8 ch, fanout 2
            int byte_ = b >> 3, j = b & 7, i = j & 3;
            c = (i & 1) * 4 + byte_; t = i >> 1; mag = (j >> 2) & 1;
        } else {                                // Fortaleza, 64 tracks
            int b32 = b & 31;
            if (b32 == 4) b32 = 8; else if (b32 == 8) b32 = 4;
            else if (b32 == 6) b32 = 10; else if (b32 == 10) b32 = 6;
            int byte_ = (b32 >> 3) + 4 * (b >> 5), j = b32 & 7, i = j & 3;
            c = (byte_ >> 2) * 8 + (i & 1) * 4 + (byte_ & 3);
            t = i >> 1; mag = (j >> 2) & 1;
        }
        (mag ? mpos : spos)[t * nchan + c] = b;
    }
    for (int i = 0; i < fanout * nchan; ++i) {
        if (spos[i] < 0 || mpos[i] < 0) {
            err = "internal error: incomplete Mark 4 bit table";
            return false;
        }
        pos[i] = (uint16_t)(spos[i] | (mpos[i] << 8));
    }
    return true;
}

inline bool m4_is_fast(int nchan, int fanout, int ft) {
    return !ft && fanout == 4 && (nchan == 4 || nchan == 8);
}

// Decode path of the standard fan-out 4 layouts (32 / 64 tracks), selectable
// with BB_TUNE_M4 for comparison runs: 2 (default) = WARP with the
// standard-layout decode (every warp store 512 contiguous bytes; C3 6.27 ->
// 6.70 TB/s, 32 tracks 6.60 -> 6.72, profiles/r2_sweep_variants.txt); 1 =
// table-driven WARP decode; 0 = per-half-word FAST decode for 8 channels
// (16 pieces of 32 B per warp store) and table-driven WARP for 4.
inline int m4_tune() {
    const char *e = getenv("BB_TUNE_M4");
    return (e && *e) ? atoi(e) : 2;
}

inline bool m4_base_geom(int nchan, int fanout, int ft, const float *levels,
                         M4Geom &g, std::string &err) {
    int ntrack;
    for (int i = 0; i < 32; ++i) g.pos[i] = 0;
    if (!m4_build_pos(nchan, fanout, ft, g.pos, ntrack, err)) return false;
    g.nchan = nchan;
    g.fanout = fanout;
    g.wordbytes = ntrack / 8;
    g.log2_nchan = ilog2_exact(nchan);
    for (int i = 0; i < 4; ++i) g.levels[i] = levels ? levels[i] : 0.f;
    g.unit_offset = nullptr;
    g.src = nullptr; g.out = nullptr; g.in = nullptr;
    g.in_elem_offset = 0;
    g.fill = 0.f;
    g.std4 = (m4_is_fast(nchan, fanout, ft) && m4_tune() == 2) ? 1u : 0u;
    return true;
}

// Decode: the per-half-word FAST path only where a row is >= 32 bytes (8
// channels); the 4-channel layout stores 16-byte pieces 64 bytes apart there
// and is faster through the WARP path.
inline bool m4_dec_fast(int nchan, int fanout, int ft) {
    return !ft && fanout == 4 && nchan == 8 && m4_tune() == 0;
}

// WARP decode needs the 8 bits of every output float4 inside one 32-bit half
// of the track word.
inline bool m4_warp_ok(const M4Geom &g) {
    const int n = g.fanout * g.nchan;
    if (n % 4) return false;
    for (int i = 0; i < n; i += 4) {
        const int half = (g.pos[i] & 0xff) >> 5;
        for (int k = 0; k < 4; ++k)
            if (((g.pos[i + k] & 0xff) >> 5) != half
                || ((g.pos[i + k] >> 8) >> 5) != half)
                return false;
    }
    return true;
}

inline void m4_warp_geom(M4Geom &g, uint32_t nframe) {
    g.log2_wordbytes = ilog2_exact(g.wordbytes);
    g.per_frame32 = g.steps * g.wordbytes / 4;
    g.total32 = g.per_frame32 * nframe;
    g.div_frame32 = make_fastdiv(g.per_frame32);
    g.nitems = (g.total32 + 31u) / 32u * 32u;         // lanes, whole warps
    for (int i = 0; i < 8; ++i) g.psel[i] = (uint8_t)(i & 3);
    if (g.wordbytes == 8) {
        int n[2] = {0, 0};
        for (int pp = 0; pp < 8; ++pp) {
            const int half = (g.pos[4 * pp] & 0xff) >> 5;
            if (n[half] < 4) g.psel[4 * half + n[half]++] = (uint8_t)pp;
        }
    }
}

// Frames API.  steps = 20000, header_steps = 160.  in_align: the bytes of one
// four-value input load (16 for float32 / float64, 8 for the 16-bit types),
// so that every input type gets the same decomposition.
inline bool plan_m4_frames(bool encode, const void *src_or_dst,
                           const int64_t *unit_offset, int64_t nframe,
                           int nchan, int fanout, int ft, const float *levels,
                           float fill, int64_t sample_start, int64_t nsample,
                           void *out, const void *in,
                           std::vector<M4Launch> &launches, std::string &err,
                           uintptr_t in_align = 16) {
    M4Geom base;
    if (!m4_base_geom(nchan, fanout, ft, levels, base, err)) return false;
    const uint32_t steps = 20000, hsteps = 160;
    const int64_t spf = (int64_t)steps * fanout;
    if (nframe < 0 || sample_start < 0 || nsample < 0
        || sample_start + nsample > nframe * spf) {
        err = "sample range outside the given frames";
        return false;
    }
    if (nsample == 0 || nframe == 0) return true;
    int mode;
    uint64_t per_frame;
    if (encode ? m4_is_fast(nchan, fanout, ft)
               : m4_dec_fast(nchan, fanout, ft)) {
        mode = M4_FAST;
        per_frame = (uint64_t)steps * (base.wordbytes / 4);
    } else if (encode && m4_warp_ok(base)
               && ((uintptr_t)src_or_dst & 3u) == 0
               && ((uintptr_t)in & (in_align - 1)) == 0) {
        mode = M4_HALF;                        // one item per 32-bit value
        per_frame = (uint64_t)steps * base.wordbytes / 4;
    } else if (encode) {
        mode = M4_GENERIC_SCALAR;              // one item per track word
        per_frame = steps;
    } else if ((sample_start * nchan) % 4 == 0 && (nsample * nchan) % 4 == 0) {
        mode = (m4_warp_ok(base) && ((uintptr_t)src_or_dst & 3u) == 0)
            ? M4_WARP : M4_GENERIC_VEC;
        per_frame = (uint64_t)spf * nchan / 4;
    } else {
        mode = M4_GENERIC_SCALAR;
        per_frame = (uint64_t)spf * nchan;
    }
    int64_t first = sample_start / spf;
    int64_t last = (sample_start + nsample + spf - 1) / spf;
    int64_t max_frames = (int64_t)(0x3fffffffull / per_frame);
    for (int64_t f0 = first; f0 < last; f0 += max_frames) {
        int64_t f1 = f0 + max_frames < last ? f0 + max_frames : last;
        M4Geom g = base;
        g.src = (const uint8_t *)src_or_dst;
        g.unit_offset = (const long long *)unit_offset + f0;
        g.out = out;
        g.in = in;
        g.in_elem_offset = (unsigned long long)(f0 * spf * nchan);
        g.row_base = f0 * spf - sample_start;
        g.nsample = nsample;
        g.nframe = (uint32_t)(f1 - f0);
        g.steps = steps;
        g.header_steps = hsteps;
        g.fill = fill;
        g.nitems = (uint32_t)(per_frame * (uint64_t)(f1 - f0));
        g.div_steps = make_fastdiv(steps);
        g.div_spf = make_fastdiv((uint32_t)spf);
        if (mode == M4_WARP) m4_warp_geom(g, g.nframe);
        if (mode == M4_HALF) {
            m4_warp_geom(g, g.nframe);
            g.nitems = g.total32;
        }
        launches.push_back({mode, g});
    }
    return true;
}

// Bare payload words (Mark4Payload.data / fromdata): no header region.
inline bool plan_m4_words(bool encode, const void *words, int64_t nword,
                          int nchan, int fanout, int ft, const float *levels,
                          float *out, const void *in,
                          std::vector<M4Launch> &launches, std::string &err) {
    M4Geom base;
    if (!m4_base_geom(nchan, fanout, ft, levels, base, err)) return false;
    if (nword < 0) { err = "nword must be >= 0"; return false; }
    const int64_t chunk = 1 << 24;             // words per launch
    for (int64_t w0 = 0; w0 < nword; w0 += chunk) {
        int64_t n = nword - w0 < chunk ? nword - w0 : chunk;
        M4Geom g = base;
        g.src = (const uint8_t *)words + w0 * base.wordbytes;
        g.unit_offset = nullptr;
        g.out = out ? out + w0 * fanout * nchan : nullptr;
        g.in = in;
        g.in_elem_offset = (unsigned long long)(w0 * fanout * nchan);
        g.row_base = 0;
        g.nsample = n * fanout;
        g.nframe = 1;
        g.steps = (uint32_t)n;
        g.header_steps = 0;
        g.div_steps = make_fastdiv((uint32_t)n);
        g.div_spf = make_fastdiv((uint32_t)(n * fanout));
        int mode;
        if (encode ? m4_is_fast(nchan, fanout, ft)
                   : m4_dec_fast(nchan, fanout, ft)) {
            mode = M4_FAST;
            g.nitems = (uint32_t)(n * (base.wordbytes / 4));
        } else if (encode && m4_warp_ok(g) && (n * base.wordbytes) % 4 == 0
                   && ((uintptr_t)g.src & 3u) == 0
                   && ((uintptr_t)in & 15u) == 0) {
            mode = M4_HALF;
            m4_warp_geom(g, 1);
            g.nitems = g.total32;
        } else if (encode) {
            mode = M4_GENERIC_SCALAR;
            g.nitems = (uint32_t)n;
        } else if (m4_warp_ok(g) && (n * base.wordbytes) % 4 == 0
                   && ((uintptr_t)g.src & 3u) == 0) {
            mode = M4_WARP;
            m4_warp_geom(g, 1);
        } else {
            mode = M4_GENERIC_VEC;             // fanout*nchan % 4 == 0 always
            g.nitems = (uint32_t)(n * fanout * nchan / 4);
        }
        launches.push_back({mode, g});
    }
    return true;
}

}  // namespace bb
