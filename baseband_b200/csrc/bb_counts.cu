// State counts of packed bit-field payloads (sm_100a): a consumer that works
// on the packed words and never materialises float32 samples in HBM.
//
// counts[bin][thread][elem][code] = number of samples of `elem` (channel, or
// re/im component of a channel) of VDIF thread `thread` whose code is `code`,
// over the valid frames of integration bin `bin`.  Codes are the bit fields of
// the payload in the reference's layout (baseband/vdif/payload.py:53-63,
// baseband/mark5b/payload.py:20-59: sample i of a word occupies bits
// [i*bps, (i+1)*bps), element index fastest), i.e. exactly what the decode
// kernels look up in the level table, so that
//     sum(decoded**2) over a bin  ==  sum_c counts[..., c] * levels[c]**2.
// Integer counts are order-independent: the result is bit-exact whatever the
// launch shape.  HBM-read bound: one pass over the packed bytes.
//
// Kernels: k_state_counts_reg (1/2 bit, <= 16 counters per word: popcounts in
// registers), k_state_counts_vert / _vert4 (more elements, 4 bit: vertical
// counters; with a word transform also Mark 4 track words,
// bb_mark4_state_counts), k_state_counts_hist (4-bit units too large for the
// 16-bit counters of _vert4), k_int8_moments (8-bit two's complement: n, sum,
// sum of squares).
#include "bb_runtime.cuh"
#include "bb_mark4_plan.h"

namespace bb {

struct CountGeom {
    const uint8_t *src;
    const long long *unit_offset;     // [nset][nthread], < 0: invalid frame
    unsigned long long *counts;       // [nbin][nthread][nelem][ncode]
    long long nset;                   // frame sets in this call
    long long set_origin;             // set 0 of this call, counted from bin 0
    long long sets_per_bin;
    long long bin_first;              // first bin this launch covers
    int nthread, nelem, split;
    uint32_t nword;                   // 32-bit words per unit payload
    uint32_t nseg;                    // register path: work items per unit
    // Mark 4 (vertical counters with a word transform): channel of every
    // two-bit field of a transformed word, per word class
    uint8_t field_elem[2][16];
};

__device__ __forceinline__ bool count_range(const CountGeom &p, long long &lo,
                                            long long &hi, long long &bin) {
    bin = p.bin_first + blockIdx.z;
    lo = bin * p.sets_per_bin - p.set_origin;
    hi = lo + p.sets_per_bin;
    if (lo < 0) lo = 0;
    if (hi > p.nset) hi = p.nset;
    return lo < hi;
}

template <int BPS, int NE>
struct ElemMask {
    // sample slots of element e within a word, one bit (the lowest of the
    // field) per slot
    static __host__ __device__ constexpr uint32_t of(int e) {
        uint32_t m = 0u;
        for (int s = e; s < 32 / BPS; s += NE) m |= 1u << (s * BPS);
        return m;
    }
};

// Register path: NE elements per word (NE * ncode <= 16 counters), counted
// with popcounts.  1 bit: c[e][0] = samples with the bit set.  2 bit: the low
// and the high bit of every field are counted separately, and the fields with
// both set: c[e][0] = n1 + n3, c[e][1] = n2 + n3, c[e][2] = n3 (n_k = samples
// with code k); the codes are separated, and code 0 found from the number of
// words seen, once per CTA at the end.
template <int BPS, int NE>
__device__ __forceinline__ void count_word(uint32_t w, uint32_t (&c)[NE][3]) {
    if (BPS == 1) {
#pragma unroll
        for (int e = 0; e < NE; ++e)
            c[e][0] += __popc(w & ElemMask<1, NE>::of(e));
    } else {
        const uint32_t lo = w & 0x55555555u, hi = (w >> 1) & 0x55555555u;
        const uint32_t both = lo & hi;
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            const uint32_t m = ElemMask<2, NE>::of(e);
            c[e][0] += __popc(lo & m);
            c[e][1] += __popc(hi & m);
            c[e][2] += __popc(both & m);
        }
    }
}

// Four words at once (one 16-byte load).  2 bit: the low-bit masks of two
// words only occupy the even bit positions, so two of them share one
// popcount (a + 2 b is a single LEA), and likewise the high-bit masks: 6
// popcounts and 3 three-input adds per 64 samples instead of 12 and 12.
template <int BPS, int NE>
__device__ __forceinline__ void count_quad(const uint4 &v,
                                           uint32_t (&c)[NE][3]) {
    if (BPS != 2) {
        count_word<BPS, NE>(v.x, c);
        count_word<BPS, NE>(v.y, c);
        count_word<BPS, NE>(v.z, c);
        count_word<BPS, NE>(v.w, c);
        return;
    }
    const uint32_t M = 0x55555555u;
    const uint32_t l0 = (v.x & M) + 2u * (v.y & M);
    const uint32_t h0 = ((v.x >> 1) & M) + 2u * ((v.y >> 1) & M);
    const uint32_t l1 = (v.z & M) + 2u * (v.w & M);
    const uint32_t h1 = ((v.z >> 1) & M) + 2u * ((v.w >> 1) & M);
    const uint32_t b0 = l0 & h0, b1 = l1 & h1;
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        const uint32_t m = ElemMask<2, NE>::of(e) * 3u;   // both words' slots
        c[e][0] += __popc(l0 & m) + __popc(l1 & m);
        c[e][1] += __popc(h0 & m) + __popc(h1 & m);
        c[e][2] += __popc(b0 & m) + __popc(b1 & m);
    }
}

constexpr int kCountBlock = 256;
constexpr uint32_t kCountSeg = 128;     // 16-byte quads per work item (4 per lane)

template <int BPS, int NE>
__global__ void __launch_bounds__(kCountBlock)
k_state_counts_reg(const CountGeom p) {
    constexpr int NCODE = 1 << BPS;
    __shared__ unsigned long long tot[NE * NCODE];
    long long lo, hi, bin;
    if (!count_range(p, lo, hi, bin)) return;
    const int t = blockIdx.y;
    if (threadIdx.x < NE * NCODE) tot[threadIdx.x] = 0ull;
    __syncthreads();
    uint32_t c[NE][3];
#pragma unroll
    for (int e = 0; e < NE; ++e) c[e][0] = c[e][1] = c[e][2] = 0u;
    uint32_t nw = 0u;
    const uint32_t nquad = p.nword / 4u;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    // The CTA owns the units of sets lo + blockIdx.x + k * split; a work item
    // is one segment (kCountSeg 16-byte quads) of one of them, taken by one
    // warp: four 16-byte loads per lane in flight before any counting, and
    // the unit offset of the warp's next item is fetched before the current
    // one is counted (the offset -> payload dependency is off the critical
    // path).  Per item the bookkeeping is one small division and one 8-byte
    // load, against 4 x ~25 counting instructions.
    const long long first = lo + blockIdx.x;
    const uint32_t nitem = first >= hi ? 0u
        : (uint32_t)((hi - first + p.split - 1) / p.split) * p.nseg;
    const long long *uo = p.unit_offset + t;
    uint32_t item = warp, g = 0u;
    long long off = -1;
    if (item < nitem) {
        const uint32_t k = item / p.nseg;
        g = item - k * p.nseg;
        off = uo[(first + (long long)k * p.split) * p.nthread];
    }
    while (item < nitem) {
        const uint32_t next = item + kCountBlock / 32;
        uint32_t g_next = 0u;
        long long off_next = -1;
        if (next < nitem) {
            const uint32_t k = next / p.nseg;
            g_next = next - k * p.nseg;
            off_next = uo[(first + (long long)k * p.split) * p.nthread];
        }
        if (off >= 0) {                              // < 0: invalid frame
            const uint8_t *base = p.src + off;
            const uint32_t *w = reinterpret_cast<const uint32_t *>(base);
            const bool last = g + 1u == p.nseg;
            uint32_t w0 = g * (kCountSeg * 4u);      // words left to do singly
            uint32_t w1 = last ? p.nword : w0 + kCountSeg * 4u;
            if ((reinterpret_cast<uintptr_t>(base) & 15u) == 0) {
                const uint4 *q = reinterpret_cast<const uint4 *>(base);
                const uint32_t i0 = g * kCountSeg + lane;
                uint4 v[kCountSeg / 32];
#pragma unroll
                for (int u = 0; u < kCountSeg / 32; ++u)
                    if (i0 + 32u * u < nquad) v[u] = q[i0 + 32u * u];
#pragma unroll
                for (int u = 0; u < kCountSeg / 32; ++u)
                    if (i0 + 32u * u < nquad) {
                        count_quad<BPS, NE>(v[u], c);
                        nw += 4u;
                    }
                w0 = last ? nquad * 4u : w1;         // the 0-3 tail words
            }
            for (uint32_t i = w0 + lane; i < w1; i += 32u) {
                count_word<BPS, NE>(w[i], c);
                nw += 1u;
            }
        }
        item = next;
        g = g_next;
        off = off_next;
    }
    // warp sums -> shared 64-bit totals -> one global atomic per counter
    const uint32_t nw_warp = __reduce_add_sync(0xffffffffu, nw);
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        uint32_t n[4];                               // per code, this warp
        const uint32_t all = nw_warp * (32 / BPS / NE);
        if (BPS == 1) {
            n[1] = __reduce_add_sync(0xffffffffu, c[e][0]);
            n[0] = all - n[1];
        } else {
            const uint32_t vl = __reduce_add_sync(0xffffffffu, c[e][0]);
            const uint32_t vh = __reduce_add_sync(0xffffffffu, c[e][1]);
            n[3] = __reduce_add_sync(0xffffffffu, c[e][2]);
            n[1] = vl - n[3];
            n[2] = vh - n[3];
            n[0] = all - n[1] - n[2] - n[3];
        }
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < NCODE; ++k)
                if (n[k])
                    atomicAdd(&tot[e * NCODE + k], (unsigned long long)n[k]);
        }
    }
    __syncthreads();
    if (threadIdx.x < NE * NCODE && tot[threadIdx.x])
        atomicAdd(p.counts + ((size_t)(bin * p.nthread + t) * NE) * NCODE
                  + threadIdx.x, tot[threadIdx.x]);
}

// General path (any power-of-two nelem, bps 1, 2 or 4): every thread keeps a
// private histogram over (slot in word, code) in shared memory -- laid out
// [counter][thread], so bank = thread and no two threads ever touch the same
// word -- and always sees words of the same class (word index mod P, P =
// words per complete sample), so that a slot is one fixed element.
constexpr int kHistBlock = 128;

template <int BPS>
__global__ void __launch_bounds__(kHistBlock)
k_state_counts_hist(const CountGeom p, int words_per_sample) {
    constexpr int NCODE = 1 << BPS, SPW = 32 / BPS, NCNT = SPW * NCODE;
    extern __shared__ uint32_t hist[];            // [NCNT][kHistBlock]
    long long lo, hi, bin;
    if (!count_range(p, lo, hi, bin)) return;
    const int t = blockIdx.y;
    // a thread's words are `stride` apart, so their class (index mod P) is
    // fixed; more classes than threads: one pass per kHistBlock classes
    const uint32_t P = (uint32_t)words_per_sample;      // a power of two
    const uint32_t stride = P > kHistBlock ? P : kHistBlock;
    const uint32_t npass = P > kHistBlock ? P / kHistBlock : 1u;
    const uint32_t lane = threadIdx.x & 31u;
    unsigned long long *out = p.counts
        + (size_t)(bin * p.nthread + t) * p.nelem * NCODE;
    for (uint32_t m = 0; m < npass; ++m) {
        const uint32_t start = threadIdx.x + kHistBlock * m;
        // (only this thread touches column threadIdx.x: no barrier needed)
        for (int c = 0; c < NCNT; ++c)
            hist[c * kHistBlock + threadIdx.x] = 0u;
        for (long long s = lo + blockIdx.x; s < hi; s += p.split) {
            const long long off = p.unit_offset[s * p.nthread + t];
            if (off < 0) continue;
            const uint32_t *w =
                reinterpret_cast<const uint32_t *>(p.src + off);
            for (uint32_t i = start; i < p.nword; i += stride) {
                const uint32_t v = w[i];
#pragma unroll
                for (int j = 0; j < SPW; ++j) {
                    const uint32_t code = (v >> (j * BPS)) & (NCODE - 1);
                    // fire-and-forget shared atomic (the column is private:
                    // atomicity is not needed, but a plain += makes every
                    // sample wait for the previous one's load-add-store)
                    atomicAdd(&hist[(j * NCODE + code) * kHistBlock
                                    + threadIdx.x], 1u);
                }
            }
        }
        // lanes of a warp that share a class add up by shuffles, then one
        // global atomic per (class, slot, code) and warp
        const uint32_t cls = start % P;
        for (int j = 0; j < SPW; ++j) {
            const uint32_t e = p.nelem >= SPW ? cls * SPW + j : j % p.nelem;
#pragma unroll
            for (int code = 0; code < NCODE; ++code) {
                uint32_t v =
                    hist[(j * NCODE + code) * kHistBlock + threadIdx.x];
                for (uint32_t o = 16; o >= P && o >= 1; o >>= 1)
                    v += __shfl_xor_sync(0xffffffffu, v, o);
                if ((P >= 32 || lane < P) && v)
                    atomicAdd(out + (size_t)e * NCODE + code,
                              (unsigned long long)v);
            }
        }
    }
}

// 1 and 2 bits with more elements than the register path holds: vertical
// counters.  The low bits of the 16 two-bit fields of a word (and the high
// bits, and the fields with both set; 1 bit: the even and the odd bits) are
// 16 one-bit indicators spaced two bits apart -- words of them can simply be
// ADDED, three at a time, into 16 two-bit fields; those are spilled into
// four-bit fields (every 3 words), those into bytes (every 15; the bytes
// live in shared memory, registers are what limits this kernel), those into
// the thread's private 32-bit counters in shared memory (every 255).  About
// 17 integer operations per word whatever the number of channels, against a
// shared-memory read-modify-write per SAMPLE in the histogram path (0.5
// TB/s).  A thread's words are `stride` apart, so a field is one fixed
// element; the codes are separated at the end as in the register path.
// Mark 4 track words -> words of sixteen two-bit codes (sign | magnitude <<
// 1), so that the vertical counters apply unchanged.  Standard fan-out 4
// layouts (32 / 64 tracks): the reference's reorder32 bit swap
// (baseband/mark4/payload.py:48-69) does exactly that.  The other layouts
// keep, per byte, four sign bits below four magnitude bits
// (mark4/payload.py:122-288): both nibbles are spread to every other bit and
// interleaved; Fortaleza first swaps track bits 4 <-> 8 and 6 <-> 10.
enum { XF_NONE = 0, XF_M4_REORDER = 1, XF_M4_NIBBLES = 2, XF_M4_FT = 3 };

__host__ __device__ __forceinline__ uint32_t m4_spread4(uint32_t x) {
    x = (x | (x << 2)) & 0x33333333u;     // nibble bits 0..3 -> 0, 1, 4, 5
    return (x | (x << 1)) & 0x55555555u;  //                   -> 0, 2, 4, 6
}

template <int XF>
__host__ __device__ __forceinline__ uint32_t m4_to_codes(uint32_t w) {
    if (XF == XF_M4_REORDER)
        return (w & 0xAA55AA55u) | ((w & 0x55005500u) >> 7)
            | ((w & 0x00AA00AAu) << 7);
    if (XF == XF_M4_FT) {
        const uint32_t t = ((w >> 4) ^ w) & 0x00000050u;
        w ^= t | (t << 4);
    }
    if (XF == XF_M4_NIBBLES || XF == XF_M4_FT)
        return m4_spread4(w & 0x0f0f0f0fu)
            | (m4_spread4((w >> 4) & 0x0f0f0f0fu) << 1);
    return w;
}

#ifndef BB_VERT_WORDS
#define BB_VERT_WORDS 15
#endif
#ifndef BB_VERT_MINB
#define BB_VERT_MINB 5
#endif
constexpr int kVertBlock = 128;
constexpr int kVertWords = BB_VERT_WORDS;   // loads in flight per thread (3 n)

template <int BPS, int XF = XF_NONE>
__global__ void __launch_bounds__(kVertBlock, BB_VERT_MINB)
k_state_counts_vert(const CountGeom p, int words_per_sample) {
    constexpr int NI = BPS == 2 ? 3 : 2;    // indicator words per data word
    constexpr int NCODE = 1 << BPS, SPW = 32 / BPS;
    constexpr uint32_t M1 = 0x55555555u, M2 = 0x33333333u, M4 = 0x0f0f0f0fu;
    constexpr uint32_t kWarps = kVertBlock / 32;
    // private columns: 32-bit counters [NI * 16] and byte fields [NI * 4]
    extern __shared__ uint32_t cnt[];       // [NI * 20][kVertBlock]
    long long lo, hi, bin;
    if (!count_range(p, lo, hi, bin)) return;
    const int t = blockIdx.y;
    // a warp takes whole units (frames are small: a CTA-wide stride would
    // leave a thread a handful of words of each); a lane's words are
    // `stride` apart, so their class (index mod P) is fixed; more classes
    // than lanes: one pass per 32 classes
    const uint32_t P = (uint32_t)words_per_sample;      // a power of two
    const uint32_t stride = P > 32u ? P : 32u;
    const uint32_t npass = P > 32u ? P / 32u : 1u;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    unsigned long long *out = p.counts
        + (size_t)(bin * p.nthread + t) * p.nelem * NCODE;
    for (uint32_t m = 0; m < npass; ++m) {
        const uint32_t start = lane + 32u * m;
        for (int c = 0; c < NI * 16; ++c)
            cnt[c * kVertBlock + threadIdx.x] = 0u;
        uint32_t *a8 = cnt + NI * 16 * kVertBlock + threadIdx.x;   // [NI * 4]
        for (int c = 0; c < NI * 4; ++c) a8[c * kVertBlock] = 0u;
        uint32_t nblock = 0u, nw = 0u;
        // field f of a2 -> field f / 2 of a4[f % 2]; field h of a4[q] ->
        // byte h / 2 of a8[2 q + h % 2]: byte g of a8[2 q + r] counts field
        // 4 g + 2 r + q.  (Rolled loops: this runs once per 255 words.)
        auto flush = [&]() {
#pragma unroll 1
            for (int c = 0; c < NI * 4; ++c) {
                const int n = c >> 2, k = c & 3;
                const uint32_t b = a8[c * kVertBlock];
                a8[c * kVertBlock] = 0u;
                uint32_t *c0 = cnt + (n * 16 + 2 * (k & 1) + (k >> 1))
                    * kVertBlock + threadIdx.x;
#pragma unroll
                for (int g = 0; g < 4; ++g)               // field 4 g + ...
                    c0[4 * g * kVertBlock] += (b >> (8 * g)) & 0xffu;
            }
            nblock = 0u;
        };
        for (long long s = lo + (long long)blockIdx.x * kWarps + warp; s < hi;
             s += (long long)p.split * kWarps) {
            const long long off = p.unit_offset[s * p.nthread + t];
            if (off < 0 || start >= p.nword) continue;
            const uint32_t *w =
                reinterpret_cast<const uint32_t *>(p.src + off);
            nw += (p.nword - start + stride - 1u) / stride;
            for (uint32_t i0 = start; i0 < p.nword;
                 i0 += kVertWords * stride) {
                uint32_t v[kVertWords];
#pragma unroll
                for (int j = 0; j < kVertWords; ++j) {
                    const uint32_t i = i0 + j * stride;
                    v[j] = i < p.nword ? w[i] : 0u;   // 0: adds nothing
                }
                if (XF != XF_NONE) {
#pragma unroll
                    for (int j = 0; j < kVertWords; ++j)
                        v[j] = m4_to_codes<XF>(v[j]);
                }
                uint32_t a4[NI][2];
#pragma unroll
                for (int n = 0; n < NI; ++n) a4[n][0] = a4[n][1] = 0u;
#pragma unroll
                for (int g = 0; g < kVertWords / 3; ++g) {
                    if (i0 + 3u * g * stride >= p.nword) break;
                    // three words: indicators add up in two-bit fields
                    const uint32_t v0 = v[3 * g], v1 = v[3 * g + 1],
                                   v2 = v[3 * g + 2];
                    const uint32_t x0 = v0 & M1, y0 = (v0 >> 1) & M1;
                    const uint32_t x1 = v1 & M1, y1 = (v1 >> 1) & M1;
                    const uint32_t x2 = v2 & M1, y2 = (v2 >> 1) & M1;
                    uint32_t a2[NI];
                    a2[0] = x0 + x1 + x2;
                    a2[1] = y0 + y1 + y2;
                    if (BPS == 2)
                        a2[NI - 1] = (x0 & y0) + (x1 & y1) + (x2 & y2);
#pragma unroll
                    for (int n = 0; n < NI; ++n) {
                        a4[n][0] += a2[n] & M2;
                        a4[n][1] += (a2[n] >> 2) & M2;
                    }
                }
                // at most 5 groups in the four-bit fields: into the bytes
#pragma unroll
                for (int n = 0; n < NI; ++n)
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        a8[(n * 4 + 2 * q) * kVertBlock] += a4[n][q] & M4;
                        a8[(n * 4 + 2 * q + 1) * kVertBlock] +=
                            (a4[n][q] >> 4) & M4;
                    }
                if (++nblock == 255u / kVertWords) flush();    // bytes full
            }
        }
        flush();
        // field f of indicator n -> sample slot; lanes that share a class
        // add up by shuffles, then global atomics (one set per warp)
        const uint32_t cls = start % P;
        uint32_t all = nw;
        for (uint32_t o = 16; o >= P && o >= 1; o >>= 1)
            all += __shfl_xor_sync(0xffffffffu, all, o);
        for (int f = 0; f < 16; ++f) {
            uint32_t c[NI];
#pragma unroll
            for (int n = 0; n < NI; ++n) {
                c[n] = cnt[(n * 16 + f) * kVertBlock + threadIdx.x];
                for (uint32_t o = 16; o >= P && o >= 1; o >>= 1)
                    c[n] += __shfl_xor_sync(0xffffffffu, c[n], o);
            }
            if (!(P >= 32u || lane < P)) continue;
            if (BPS == 2) {
                const uint32_t e = XF != XF_NONE ? p.field_elem[cls & 1u][f]
                    : p.nelem >= SPW ? cls * SPW + f : f % p.nelem;
                const uint32_t n3 = c[NI - 1], n1 = c[0] - n3, n2 = c[1] - n3;
                // Mark 4 counts are indexed 2 * sign + magnitude, as its level
                // table is: fields are sign | magnitude << 1, so 1 <-> 2
                const uint32_t nk[4] = {all - n1 - n2 - n3,
                                        XF != XF_NONE ? n2 : n1,
                                        XF != XF_NONE ? n1 : n2, n3};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (nk[k])
                        atomicAdd(out + (size_t)e * NCODE + k % NCODE,
                                  (unsigned long long)nk[k]);
            } else {
#pragma unroll
                for (int n = 0; n < 2; ++n) {
                    const uint32_t slot = 2u * f + n;
                    const uint32_t e = p.nelem >= SPW ? cls * SPW + slot
                        : slot % p.nelem;
                    if (all - c[n])
                        atomicAdd(out + (size_t)e * NCODE,
                                  (unsigned long long)(all - c[n]));
                    if (c[n])
                        atomicAdd(out + (size_t)e * NCODE + 1 % NCODE,
                                  (unsigned long long)c[n]);
                }
            }
        }
    }
}

// 4 bits: the same idea with one indicator per code.  The four bit planes of
// the eight nibbles (and their complements) give the eight minterms of the
// low three bits with one LOP3 each and from those the 15 codes above zero
// with one more; an indicator is 8 one-bit flags four bits apart, so 15
// words of them add up in nibble fields, which are spilled into byte fields
// (shared memory) and those, every 255 words, into the private counters.
// ~55 integer operations per word against eight shared-memory atomics.
constexpr int kVert4Block = 128;

__global__ void __launch_bounds__(kVert4Block, 5)
k_state_counts_vert4(const CountGeom p, int words_per_sample) {
    constexpr int NI = 15, NCODE = 16, SPW = 8, NW = 15;
    constexpr uint32_t M = 0x11111111u, M4 = 0x0f0f0f0fu;
    constexpr uint32_t kWarps = kVert4Block / 32;
    // private columns: pairs of 16-bit counters [NI * 4] (the launcher keeps
    // a lane below 2^16 words: shared memory is what limits the number of
    // resident warps here), byte fields [NI * 2]
    extern __shared__ uint32_t cnt[];       // [NI * 6][kVert4Block]
    long long lo, hi, bin;
    if (!count_range(p, lo, hi, bin)) return;
    const int t = blockIdx.y;
    const uint32_t P = (uint32_t)words_per_sample;      // a power of two
    const uint32_t stride = P > 32u ? P : 32u;
    const uint32_t npass = P > 32u ? P / 32u : 1u;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    unsigned long long *out = p.counts
        + (size_t)(bin * p.nthread + t) * p.nelem * NCODE;
    uint32_t *a8 = cnt + NI * 4 * kVert4Block + threadIdx.x;       // [NI * 2]
    for (uint32_t m = 0; m < npass; ++m) {
        const uint32_t start = lane + 32u * m;
        for (int c = 0; c < NI * 6; ++c)
            cnt[c * kVert4Block + threadIdx.x] = 0u;
        uint32_t nblock = 0u, nw = 0u;
        // byte g of a8[2 c + r] counts nibble field 2 g + r of indicator c;
        // cnt[4 c + g] holds fields 2 g (low half) and 2 g + 1 (high half)
        auto flush = [&]() {
#pragma unroll 1
            for (int c = 0; c < NI; ++c) {
                const uint32_t b0 = a8[(2 * c) * kVert4Block];
                const uint32_t b1 = a8[(2 * c + 1) * kVert4Block];
                a8[(2 * c) * kVert4Block] = 0u;
                a8[(2 * c + 1) * kVert4Block] = 0u;
                uint32_t *c0 = cnt + 4 * c * kVert4Block + threadIdx.x;
#pragma unroll
                for (int g = 0; g < 4; ++g)
                    c0[g * kVert4Block] += ((b0 >> (8 * g)) & 0xffu)
                        | (((b1 >> (8 * g)) & 0xffu) << 16);
            }
            nblock = 0u;
        };
        for (long long s = lo + (long long)blockIdx.x * kWarps + warp; s < hi;
             s += (long long)p.split * kWarps) {
            const long long off = p.unit_offset[s * p.nthread + t];
            if (off < 0 || start >= p.nword) continue;
            const uint32_t *w =
                reinterpret_cast<const uint32_t *>(p.src + off);
            nw += (p.nword - start + stride - 1u) / stride;
            for (uint32_t i0 = start; i0 < p.nword; i0 += NW * stride) {
                uint32_t v[NW];
#pragma unroll
                for (int j = 0; j < NW; ++j) {
                    const uint32_t i = i0 + j * stride;
                    // past the end: code 0 everywhere, which is not counted
                    v[j] = i < p.nword ? w[i] : 0u;
                }
                uint32_t a4[NI];
#pragma unroll
                for (int c = 0; c < NI; ++c) a4[c] = 0u;
#pragma unroll
                for (int j = 0; j < NW; ++j) {
                    if (i0 + (uint32_t)j * stride >= p.nword) break;
                    const uint32_t x = v[j];
                    const uint32_t p0 = x & M, p1 = (x >> 1) & M;
                    const uint32_t p2 = (x >> 2) & M, p3 = (x >> 3) & M;
                    const uint32_t n0 = p0 ^ M, n1 = p1 ^ M, n2 = p2 ^ M,
                                   n3 = p3 ^ M;
                    uint32_t mt[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        mt[k] = ((k & 1) ? p0 : n0) & ((k & 2) ? p1 : n1)
                            & ((k & 4) ? p2 : n2);
#pragma unroll
                    for (int c = 1; c < 16; ++c)
                        a4[c - 1] += mt[c & 7] & ((c & 8) ? p3 : n3);
                }
                // at most 15 in the nibble fields: into the bytes
#pragma unroll
                for (int c = 0; c < NI; ++c) {
                    a8[(2 * c) * kVert4Block] += a4[c] & M4;
                    a8[(2 * c + 1) * kVert4Block] += (a4[c] >> 4) & M4;
                }
                if (++nblock == 255u / NW) flush();           // bytes full
            }
        }
        flush();
        // nibble field h of indicator c - 1 -> (sample slot h, code c); lanes
        // that share a class add up by shuffles, then global atomics
        const uint32_t cls = start % P;
        uint32_t all = nw;
        for (uint32_t o = 16; o >= P && o >= 1; o >>= 1)
            all += __shfl_xor_sync(0xffffffffu, all, o);
        for (int h = 0; h < SPW; ++h) {
            const uint32_t e = p.nelem >= SPW ? cls * SPW + h : h % p.nelem;
            uint32_t rest = all;
            for (int c = 1; c < NCODE; ++c) {
                uint32_t n = (cnt[((c - 1) * 4 + h / 2) * kVert4Block
                                  + threadIdx.x] >> (16 * (h & 1))) & 0xffffu;
                for (uint32_t o = 16; o >= P && o >= 1; o >>= 1)
                    n += __shfl_xor_sync(0xffffffffu, n, o);
                rest -= n;
                if ((P >= 32u || lane < P) && n)
                    atomicAdd(out + (size_t)e * NCODE + c,
                              (unsigned long long)n);
            }
            if ((P >= 32u || lane < P) && rest)
                atomicAdd(out + (size_t)e * NCODE, (unsigned long long)rest);
        }
    }
}

// 8-bit two's-complement samples (GUPPI, DADA): count, sum and sum of squares
// per element instead of a 256-bin histogram -- what power, mean and variance
// need, still exact integers.  A word holds four samples: each byte is
// sign-extended with one permute, added to a 32-bit sum (two words per
// three-input add) and squared into a 32-bit sum with one multiply-add; the
// partial sums are folded into 64-bit totals long before they can overflow.
// Ten integer operations per word.  (A first version used dp4a against byte
// masks -- eight dp4a per word -- and stopped at 1.5 TB/s: dp4a issues at a
// fraction of the integer rate.)  As in
// the histogram path a thread only ever sees words of one class (word index
// mod P, P = words per complete sample), so a byte lane is one fixed element.
struct MomAcc {
    // a 32-bit partial sum of squares holds 2^32 / 2^14 words
    static constexpr uint32_t kFold = (1u << 18) - 64u;
    int s[4] = {0, 0, 0, 0};
    uint32_t q[4] = {0u, 0u, 0u, 0u}, pend = 0u;
    long long sum[4] = {0, 0, 0, 0}, sq[4] = {0, 0, 0, 0}, nw = 0;

    __device__ __forceinline__ void word(uint32_t v) {
        // byte b sign-extended: one permute with sign replication (or shift)
        const int x0 = sext<0x8880u>(v), x1 = sext<0x9991u>(v);
        const int x2 = sext<0xaaa2u>(v), x3 = (int)v >> 24;
        s[0] += x0;
        s[1] += x1;
        s[2] += x2;
        s[3] += x3;
        square_add(q[0], (uint32_t)x0);
        square_add(q[1], (uint32_t)x1);
        square_add(q[2], (uint32_t)x2);
        square_add(q[3], (uint32_t)x3);
        pend += 1u;
    }
    // prmt with bit 3 of a selector nibble set replicates the sign of the
    // chosen byte (the __byte_perm intrinsic only passes three bits)
    template <uint32_t SEL>
    static __device__ __forceinline__ int sext(uint32_t v) {
        int x;
        asm("prmt.b32 %0, %1, 0, %2;" : "=r"(x) : "r"(v), "n"(SEL));
        return x;
    }
    // q += x * x as one IMAD, spelled out: left to itself the compiler gathers
    // the bytes of four words with shifts and permutes to feed a dp4a, which
    // is the slow instruction this formulation avoids.
    static __device__ __forceinline__ void square_add(uint32_t &q, uint32_t x) {
        asm("mad.lo.u32 %0, %1, %1, %0;" : "+r"(q) : "r"(x));
    }
    __device__ __forceinline__ void fold() {
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            sum[b] += s[b];
            sq[b] += q[b];
            s[b] = 0;
            q[b] = 0u;
        }
        nw += pend;
        pend = 0u;
    }
    __device__ __forceinline__ void finish() { fold(); }
};

template <int U>                        // loads in flight per thread
__global__ void __launch_bounds__(kCountBlock)
k_int8_moments(const CountGeom p, int words_per_sample) {
    long long lo, hi, bin;
    if (!count_range(p, lo, hi, bin)) return;
    const int t = blockIdx.y;
    MomAcc a;
    for (long long s = lo + blockIdx.x; s < hi; s += p.split) {
        const long long off = p.unit_offset[s * p.nthread + t];
        if (off < 0) continue;
        const uint8_t *base = p.src + off;
        const uint32_t *w = reinterpret_cast<const uint32_t *>(base);
        uint32_t first = 0u;             // words not taken by the vector pass
        if (words_per_sample == 1
            && (reinterpret_cast<uintptr_t>(base) & 15u) == 0) {
            // every word is of the same class: 16-byte loads
            const uint4 *q4 = reinterpret_cast<const uint4 *>(base);
            const uint32_t nquad = p.nword / 4u;
            for (uint32_t i0 = threadIdx.x; i0 < nquad;
                 i0 += U * kCountBlock) {
                uint4 v[U];
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (i0 + u * kCountBlock < nquad)
                        v[u] = q4[i0 + u * kCountBlock];
                if (a.pend > MomAcc::kFold) a.fold();
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (i0 + u * kCountBlock < nquad) {
                        a.word(v[u].x);
                        a.word(v[u].y);
                        a.word(v[u].z);
                        a.word(v[u].w);
                    }
            }
            first = nquad * 4u;
        }
        // a thread's words are kCountBlock apart: the class (index mod P,
        // P a power of two <= kCountBlock) stays the same
        for (uint32_t i0 = first + threadIdx.x; i0 < p.nword;
             i0 += U * kCountBlock) {
            uint32_t v[U];
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (i0 + u * kCountBlock < p.nword)
                    v[u] = w[i0 + u * kCountBlock];
            if (a.pend > MomAcc::kFold) a.fold();
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (i0 + u * kCountBlock < p.nword) a.word(v[u]);
        }
    }
    a.finish();
    const long long nw = a.nw;
    long long (&sum)[4] = a.sum, (&sq)[4] = a.sq;
    const int P = words_per_sample;               // power of two <= block
    const int cls = threadIdx.x % P;
    const uint32_t lane = threadIdx.x & 31u;
    unsigned long long *out = p.counts
        + (size_t)(bin * p.nthread + t) * p.nelem * 3;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        long long v[3] = {nw, sum[b], sq[b]};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            for (int o = 16; o >= P && o >= 1; o >>= 1)
                v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
        }
        if (P >= 32 || lane < (uint32_t)P) {
            const int e = p.nelem >= 4 ? cls * 4 + b : b % p.nelem;
#pragma unroll
            for (int k = 0; k < 3; ++k)
                if (v[k])
                    atomicAdd(out + (size_t)e * 3 + k,
                              (unsigned long long)v[k]);
        }
    }
}

// 8-bit payloads of any encoding: a 256-bin histogram of the stored byte per
// (bin, thread, element); what a byte means is left to the host's level
// table.  A CTA counts one window of elements (a `ww`-word stretch of every
// sample: all of it up to 64 elements, 64 elements beyond) over every
// split-th segment of its (bin, thread), in shared-memory counters laid out
// [byte][element in window][replica]: `nrep` copies, lane l writing copy
// l % nrep, so that nwin_elem * nrep = 64 (32 for one element) and the
// table is 64 KiB whatever the geometry.  On the 16-byte path every lane of
// a warp owns a different (element, replica) slot at every step -- a quad's
// 16 bytes are taken in an order rotated per lane -- and since the slot
// stride is the whole row of a byte value, the bank is the slot's: no two
// lanes of a warp hit the same bank, however narrow the data (same-address
// atomics would otherwise serialise on Gaussian noise that spans a handful
// of codes).  Units that are not 16-byte aligned take single words, where
// lanes 16 apart can share a slot (slower, still exact).  A work item is a
// segment of 128 16-byte quads of one unit, taken by one warp: four loads
// per lane in flight, the next item's unit offset fetched ahead.  The
// segments of a bin are dealt out to its CTAs one by one, so a single large
// unit (a DADA chunk piece) is spread over the GPU too.  Counters are 32
// bit and read out once, at the end: the launcher gives no CTA more than
// kByteMaxItems segments (2 GiB), so none can wrap.
struct ByteGeom {
    const uint8_t *src;
    const long long *unit_offset;     // [nset][nthread], < 0: invalid frame
    unsigned long long *counts;       // [nbin][nthread][nelem][256]
    long long nset, set_origin, sets_per_bin, bin_first;
    int nthread, nelem, split;
    uint32_t nwin;                    // element windows (grid.x = split * nwin)
    uint32_t lg_p, lg_ww;             // log2 words per sample, per window
    uint32_t ne;                      // elements per window
    uint32_t nrep;                    // replicas (lane l -> l % nrep)
    uint32_t nq;                      // window words per unit
    uint32_t nseg;                    // work items per unit
};

constexpr int kByteBlock = 256;
constexpr int kByteCounters = 256 * 64;
constexpr uint32_t kByteSegQuads = 128;          // 4 quads per lane
constexpr int64_t kByteMaxItems = 1ll << 20;     // x 2 KiB = 2 GiB per CTA

// 16 bytes rotated down by `rot` bytes: byte k of the result is byte
// (k + rot) & 15 of v
__device__ __forceinline__ void rotate16(const uint4 &v, uint32_t rot,
                                         uint32_t (&o)[4]) {
    uint32_t a0 = v.x, a1 = v.y, a2 = v.z, a3 = v.w;
    if (rot & 4u) { const uint32_t t = a0; a0 = a1; a1 = a2; a2 = a3; a3 = t; }
    if (rot & 8u) {
        uint32_t t = a0; a0 = a2; a2 = t;
        t = a1; a1 = a3; a3 = t;
    }
    const uint32_t sh = (rot & 3u) * 8u;
    o[0] = __funnelshift_r(a0, a1, sh);
    o[1] = __funnelshift_r(a1, a2, sh);
    o[2] = __funnelshift_r(a2, a3, sh);
    o[3] = __funnelshift_r(a3, a0, sh);
}

__global__ void __launch_bounds__(kByteBlock, 3)
k_byte_counts(const ByteGeom p) {
    extern __shared__ uint32_t hist[];          // [256][ne][nrep]
    const long long bin = p.bin_first + blockIdx.z;
    long long lo = bin * p.sets_per_bin - p.set_origin;
    long long hi = lo + p.sets_per_bin;
    if (lo < 0) lo = 0;
    if (hi > p.nset) hi = p.nset;
    if (lo >= hi) return;
    const int t = blockIdx.y;
    const uint32_t win = blockIdx.x % p.nwin;
    const long long sx = blockIdx.x / p.nwin;         // this CTA's share
    const uint32_t ww = 1u << p.lg_ww, w0 = win * ww;
    const uint32_t row = p.ne * p.nrep;               // counters per byte value
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t r = lane % p.nrep;
    for (uint32_t i = threadIdx.x; i < 256u * row; i += kByteBlock) hist[i] = 0u;
    // slot (element * nrep + replica) of every step: a lane's quads all
    // start at window word (4 lane) mod ww, i.e. element (16 lane) mod ne,
    // its single words at window word lane mod ww
    const uint32_t rot = p.nrep == 1u
        ? ((lane >> 2) << 1 | (lane >> 1 & 1u)) & 15u : (lane / p.nrep) & 15u;
    uint32_t colq[16], colw[4];
#pragma unroll
    for (int k = 0; k < 16; ++k)
        colq[k] = ((16u * lane + ((k + rot) & 15u)) % p.ne) * p.nrep + r;
#pragma unroll
    for (int b = 0; b < 4; ++b)
        colw[b] = ((4u * lane + b) % p.ne) * p.nrep + r;
    __syncthreads();

    auto flush = [&]() {
        // consecutive threads read consecutive counters (no bank conflict);
        // the nrep replicas of a slot sit in adjacent lanes
        unsigned long long *out = p.counts
            + ((size_t)(bin * p.nthread + t) * p.nelem + (size_t)win * p.ne)
                * 256u;
        for (uint32_t i = threadIdx.x; i < 256u * row; i += kByteBlock) {
            uint32_t n = hist[i];
            hist[i] = 0u;
            for (uint32_t o = p.nrep >> 1; o >= 1u; o >>= 1)
                n += __shfl_xor_sync(0xffffffffu, n, o);
            if (lane % p.nrep == 0u && n) {
                const uint32_t v = i / row, e = (i % row) / p.nrep;
                atomicAdd(out + (size_t)e * 256u + v, (unsigned long long)n);
            }
        }
    };

    // window word q of a unit -> word index in the payload
    auto word_at = [&](uint32_t q) {
        return ((q >> p.lg_ww) << p.lg_p) + w0 + (q & (ww - 1u));
    };
    auto count_word = [&](uint32_t v) {
#pragma unroll
        for (int b = 0; b < 4; ++b)
            atomicAdd(&hist[((v >> (8 * b)) & 0xffu) * row + colw[b]], 1u);
    };
    // segments j = sx + split * item of the bin's (hi - lo) * nseg; the
    // launcher keeps nitem <= kByteMaxItems
    const long long jn = (hi - lo) * p.nseg;
    const uint32_t nitem = sx >= jn ? 0u
        : (uint32_t)((jn - sx + p.split - 1) / p.split);
    const long long *uo = p.unit_offset + t;
    // a warp's items are split * 8 segments apart: (unit k, segment g) of
    // the next one by an add with carry, no division per item
    const long long step = (long long)p.split * (kByteBlock / 32);
    const long long dk = step / p.nseg;
    const uint32_t dg = (uint32_t)(step - dk * p.nseg);
    const long long j0 = sx + (long long)p.split * warp;
    long long k = j0 / p.nseg;
    uint32_t g = (uint32_t)(j0 - k * p.nseg);
    uint32_t item = warp;
    long long off = item < nitem ? uo[(lo + k) * p.nthread] : -1;
    const uint32_t nquad = p.nq / 4u;
    while (item < nitem) {
        const uint32_t next = item + kByteBlock / 32;
        uint32_t g_next = g + dg;
        long long k_next = k + dk;
        if (g_next >= p.nseg) {
            g_next -= p.nseg;
            ++k_next;
        }
        const long long off_next =
            next < nitem ? uo[(lo + k_next) * p.nthread] : -1;
        if (off >= 0) {                              // < 0: invalid frame
            const uint8_t *base = p.src + off;
            const uint32_t *w = reinterpret_cast<const uint32_t *>(base);
            const bool last = g + 1u == p.nseg;
            const uint32_t q0 = g * kByteSegQuads * 4u;
            uint32_t q1 = last ? p.nq : q0 + kByteSegQuads * 4u;
            uint32_t qs = q0;                        // words left to do singly
            if ((reinterpret_cast<uintptr_t>(base) & 15u) == 0) {
                // four window words in a row are adjacent in memory: the
                // window is either a whole sample or a multiple of 4 words
                const uint4 *q = reinterpret_cast<const uint4 *>(base);
                const uint32_t i0 = g * kByteSegQuads + lane;
                uint4 v[kByteSegQuads / 32];
#pragma unroll
                for (int u = 0; u < kByteSegQuads / 32; ++u)
                    if (i0 + 32u * u < nquad)
                        v[u] = q[word_at(4u * (i0 + 32u * u)) >> 2];
#pragma unroll
                for (int u = 0; u < kByteSegQuads / 32; ++u)
                    if (i0 + 32u * u < nquad) {
                        uint32_t o[4];
                        rotate16(v[u], rot, o);
#pragma unroll
                        for (int k = 0; k < 16; ++k)
                            atomicAdd(&hist[((o[k >> 2] >> (8 * (k & 3)))
                                             & 0xffu) * row + colq[k]], 1u);
                    }
                qs = last ? nquad * 4u : q1;         // the 0-3 tail words
            }
            // unaligned units (and the tail): single words, 16 per lane in
            // flight; a lane's words stay at window word lane mod ww
            for (uint32_t i0 = qs + lane; i0 < q1; i0 += 16u * 32u) {
                uint32_t v[16];
#pragma unroll
                for (int u = 0; u < 16; ++u)
                    if (i0 + 32u * u < q1) v[u] = w[word_at(i0 + 32u * u)];
#pragma unroll
                for (int u = 0; u < 16; ++u)
                    if (i0 + 32u * u < q1) count_word(v[u]);
            }
        }
        item = next;
        g = g_next;
        k = k_next;
        off = off_next;
    }
    __syncthreads();
    flush();
}

template <int BPS, int NE>
static void launch_reg(const CountGeom &g, dim3 grid, cudaStream_t s) {
    k_state_counts_reg<BPS, NE><<<grid, kCountBlock, 0, s>>>(g);
}

template <int BPS>
static int launch_hist(const CountGeom &g, dim3 grid, int P, cudaStream_t s) {
    constexpr int NCNT = (32 / BPS) * (1 << BPS);
    const size_t smem = (size_t)NCNT * kHistBlock * sizeof(uint32_t);
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(
            k_state_counts_hist<BPS>,
            cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return check_cuda(e, "bb_state_counts (smem)");
        attr_set = true;
    }
    k_state_counts_hist<BPS><<<grid, kHistBlock, smem, s>>>(g, P);
    return BB_OK;
}

}  // namespace bb

using namespace bb;

// CTAs per SM a launch aims at (development tunables BB_TUNE_COUNT_DEPTH,
// BB_TUNE_VERT_DEPTH; defaults swept with tools/sweep_counts.py).  The
// vertical-counter kernel has a fixed cost per CTA (zeroing and reading out 60
// shared-memory words per thread, 90 at 4 bit, and its read-out is ~50
// atomics per thread, 120 at 4 bit): 16 measured best at 1/2 bit, 8 at 4 bit.
static int count_depth(bool vert = false, int bps = 2) {
    const char *e = getenv(vert ? "BB_TUNE_VERT_DEPTH" : "BB_TUNE_COUNT_DEPTH");
    return (e && *e && atoi(e) > 0) ? atoi(e) : !vert ? 24 : bps == 4 ? 8 : 16;
}

// The integration bins a call touches, and how many CTAs each (bin, grid
// row) gets: enough to fill the GPU `want` CTAs deep, at most `most` (one
// per set, or per work item, of a bin).
struct BinPlan {
    int64_t b0, nb, per_bin;

    int64_t split_for(int64_t want, int64_t rows, int64_t most) const {
        int64_t split = (want + nb * rows - 1) / (nb * rows);
        if (split > most) split = most;
        if (split < 1) split = 1;
        if (split > 65535) split = 65535;
        return split;
    }
};

static bool plan_bins(int64_t nset, int64_t set_origin, int64_t sets_per_bin,
                      int64_t nbin, BinPlan &bp) {
    bp.b0 = set_origin / sets_per_bin;
    const int64_t b1 = (set_origin + nset - 1) / sets_per_bin;    // inclusive
    bp.nb = b1 - bp.b0 + 1;
    bp.per_bin = sets_per_bin < nset ? sets_per_bin : nset;
    return b1 < nbin;
}

extern "C" int bb_state_counts(
    const void *src, const int64_t *unit_offset, int64_t nset, int32_t nthread,
    int64_t payload_nbytes, int32_t bps, int32_t nelem, int64_t set_origin,
    int64_t sets_per_bin, uint64_t *counts, int64_t nbin, void *stream) {
    if (!src || !unit_offset || !counts)
        return set_error(BB_ERR_ARGUMENT, "null pointer");
    if (!(bps == 1 || bps == 2 || bps == 4))
        return set_error(BB_ERR_UNSUPPORTED,
                         "state counts exist for 1, 2 and 4 bits per sample");
    if (nset < 0 || nthread < 1 || nthread > 65535 || nelem < 1
        || (nelem & (nelem - 1)) || payload_nbytes <= 0 || (payload_nbytes & 3)
        || set_origin < 0 || sets_per_bin < 1 || nbin < 1)
        return set_error(BB_ERR_ARGUMENT, "bad geometry (nelem must be a "
                         "power of two, payload a multiple of 4 bytes)");
    if (!aligned(src, 4))
        return set_error(BB_ERR_ALIGNMENT, "src must be 4-byte aligned");
    if (payload_nbytes / 4 > 0x7fffffff)
        return set_error(BB_ERR_ARGUMENT, "payload too large");
    if ((payload_nbytes * 8) % ((int64_t)bps * nelem))
        return set_error(BB_ERR_ARGUMENT,
                         "payload does not hold whole samples");
    if (nset == 0) return BB_OK;
    const int64_t b0 = set_origin / sets_per_bin;
    const int64_t b1 = (set_origin + nset - 1) / sets_per_bin;     // inclusive
    if (b1 >= nbin)
        return set_error(BB_ERR_ARGUMENT, "sets run past the last bin");
    const int spw = 32 / bps, ncode = 1 << bps;
    const bool reg = bps <= 2 && nelem <= spw && nelem * ncode <= 16;
    const int P = nelem > spw ? nelem / spw : 1;
    CountGeom g;
    g.src = (const uint8_t *)src;
    g.unit_offset = (const long long *)unit_offset;
    g.counts = (unsigned long long *)counts;
    g.nset = nset;
    g.set_origin = set_origin;
    g.sets_per_bin = sets_per_bin;
    g.nthread = nthread;
    g.nelem = nelem;
    g.nword = (uint32_t)(payload_nbytes / 4);
    // CTAs per (bin, thread): enough to fill the GPU 24 deep, at most one
    // per set of a bin, and few enough words each that 32-bit counters hold
    const int64_t nb = b1 - b0 + 1;
    const int64_t per_bin = sets_per_bin < nset ? sets_per_bin : nset;
    const int64_t want = (int64_t)count_depth(!reg, bps) * sm_count();
    int64_t split = (want + nb * nthread - 1) / (nb * nthread);
    int64_t need = (per_bin * (int64_t)g.nword + (1ll << 26) - 1)
        / (1ll << 26);
    bool hist4 = false;
    if (split < need) split = need;
    if (split > per_bin) split = per_bin;
    // register path: a warp takes a segment of a unit, so a CTA wants at
    // least one segment per warp
    g.nseg = (g.nword / 4u + kCountSeg - 1u) / kCountSeg;
    if (g.nseg < 1u) g.nseg = 1u;
    if (reg) {
        const int64_t full = per_bin * g.nseg / (kCountBlock / 32);
        if (split > full && full >= need) split = full;
    } else {                               // vertical counters: a unit per warp
        if (bps == 4) {
            // 16-bit counters: a lane must stay below 2^16 words
            const int64_t lane_words = ((int64_t)g.nword + 31) / 32;
            const int64_t units = 60000 / lane_words;     // per warp
            if (units < 1) {
                hist4 = true;              // huge units: histogram kernel
            } else {
                const int64_t need4 = (per_bin + units * (kVert4Block / 32) - 1)
                    / (units * (kVert4Block / 32));
                if (need4 > 65535) hist4 = true;
                else if (need4 > need) need = need4;
                if (split < need) split = need;
            }
        }
        const int64_t full = per_bin / ((bps == 4 ? kVert4Block : kVertBlock) / 32);
        if (split > full && full >= need) split = full;
    }
    if (split < 1) split = 1;
    if (split > 65535) split = 65535;
    g.split = (int)split;
    cudaStream_t s = as_stream(stream);
    for (int64_t z0 = 0; z0 < nb; z0 += 65535) {
        const int64_t nz = nb - z0 < 65535 ? nb - z0 : 65535;
        g.bin_first = b0 + z0;
        dim3 grid((unsigned)split, (unsigned)nthread, (unsigned)nz);
        if (reg) {
            if (bps == 1) {
                if (nelem == 1) launch_reg<1, 1>(g, grid, s);
                else if (nelem == 2) launch_reg<1, 2>(g, grid, s);
                else if (nelem == 4) launch_reg<1, 4>(g, grid, s);
                else launch_reg<1, 8>(g, grid, s);
            } else {
                if (nelem == 1) launch_reg<2, 1>(g, grid, s);
                else if (nelem == 2) launch_reg<2, 2>(g, grid, s);
                else launch_reg<2, 4>(g, grid, s);
            }
        } else {
            int rc = BB_OK;
            if (bps == 4 && (hist4 || getenv("BB_TUNE_COUNT_HIST4"))) {
                rc = launch_hist<4>(g, grid, P, s);       // the first version
            } else if (bps == 4) {
                const size_t smem = (size_t)15 * 6 * kVert4Block
                    * sizeof(uint32_t);
                static bool attr_set = false;
                if (!attr_set) {
                    rc = check_cuda(cudaFuncSetAttribute(
                        k_state_counts_vert4,
                        cudaFuncAttributeMaxDynamicSharedMemorySize,
                        (int)smem), "bb_state_counts (smem)");
                    attr_set = rc == BB_OK;
                }
                if (rc == BB_OK)
                    k_state_counts_vert4<<<grid, kVert4Block, smem, s>>>(g, P);
            } else {
                const size_t smem = (size_t)(bps == 2 ? 3 : 2) * 20
                    * kVertBlock * sizeof(uint32_t);
                if (bps == 2)
                    k_state_counts_vert<2><<<grid, kVertBlock, smem, s>>>(g, P);
                else
                    k_state_counts_vert<1><<<grid, kVertBlock, smem, s>>>(g, P);
            }
            if (rc != BB_OK) return rc;
        }
        BB_CHECK_LAUNCH("bb_state_counts");
    }
    return BB_OK;
}

extern "C" int bb_int8_moments(
    const void *src, const int64_t *unit_offset, int64_t nset, int32_t nthread,
    int64_t payload_nbytes, int32_t nelem, int64_t set_origin,
    int64_t sets_per_bin, int64_t *moments, int64_t nbin, void *stream) {
    if (!src || !unit_offset || !moments)
        return set_error(BB_ERR_ARGUMENT, "null pointer");
    if (nset < 0 || nthread < 1 || nthread > 65535 || nelem < 1
        || (nelem & (nelem - 1)) || payload_nbytes <= 0 || (payload_nbytes & 3)
        || payload_nbytes % nelem || set_origin < 0 || sets_per_bin < 1
        || nbin < 1)
        return set_error(BB_ERR_ARGUMENT, "bad geometry (nelem must be a "
                         "power of two, payload whole samples and words)");
    if (!aligned(src, 4))
        return set_error(BB_ERR_ALIGNMENT, "src must be 4-byte aligned");
    if (payload_nbytes / 4 > 0x7fffffff)
        return set_error(BB_ERR_ARGUMENT, "payload too large");
    const int P = nelem > 4 ? nelem / 4 : 1;
    if (P > kCountBlock)
        return set_error(BB_ERR_UNSUPPORTED,
                         "too many elements per sample for moments");
    if (nset == 0) return BB_OK;
    BinPlan bp;
    if (!plan_bins(nset, set_origin, sets_per_bin, nbin, bp))
        return set_error(BB_ERR_ARGUMENT, "sets run past the last bin");
    CountGeom g;
    g.src = (const uint8_t *)src;
    g.unit_offset = (const long long *)unit_offset;
    g.counts = (unsigned long long *)moments;
    g.nset = nset;
    g.set_origin = set_origin;
    g.sets_per_bin = sets_per_bin;
    g.nthread = nthread;
    g.nelem = nelem;
    g.nword = (uint32_t)(payload_nbytes / 4);
    const int64_t split = bp.split_for((int64_t)count_depth() * sm_count(),
                                       nthread, bp.per_bin);
    g.split = (int)split;
    for (int64_t z0 = 0; z0 < bp.nb; z0 += 65535) {
        const int64_t nz = bp.nb - z0 < 65535 ? bp.nb - z0 : 65535;
        g.bin_first = bp.b0 + z0;
        dim3 grid((unsigned)split, (unsigned)nthread, (unsigned)nz);
        const char *e_u = getenv("BB_TUNE_MOM_U");
        const int u = (e_u && *e_u) ? atoi(e_u) : 4;
        if (u == 8)
            k_int8_moments<8><<<grid, kCountBlock, 0, as_stream(stream)>>>(g, P);
        else if (u == 2)
            k_int8_moments<2><<<grid, kCountBlock, 0, as_stream(stream)>>>(g, P);
        else
            k_int8_moments<4><<<grid, kCountBlock, 0, as_stream(stream)>>>(g, P);
        BB_CHECK_LAUNCH("bb_int8_moments");
    }
    return BB_OK;
}

extern "C" int bb_byte_counts(
    const void *src, const int64_t *unit_offset, int64_t nset, int32_t nthread,
    int64_t payload_nbytes, int32_t nelem, int64_t set_origin,
    int64_t sets_per_bin, uint64_t *counts, int64_t nbin, void *stream) {
    if (!src || !unit_offset || !counts)
        return set_error(BB_ERR_ARGUMENT, "null pointer");
    if (nset < 0 || nthread < 1 || nthread > 65535 || nelem < 1
        || (nelem & (nelem - 1)) || payload_nbytes <= 0 || (payload_nbytes & 3)
        || payload_nbytes % nelem || set_origin < 0 || sets_per_bin < 1
        || nbin < 1)
        return set_error(BB_ERR_ARGUMENT, "bad geometry (nelem must be a "
                         "power of two, payload whole samples and words)");
    if (!aligned(src, 4))
        return set_error(BB_ERR_ALIGNMENT, "src must be 4-byte aligned");
    if (payload_nbytes / 4 > 0x7fffffff)
        return set_error(BB_ERR_ARGUMENT, "payload too large");
    if (nset == 0) return BB_OK;
    BinPlan bp;
    if (!plan_bins(nset, set_origin, sets_per_bin, nbin, bp))
        return set_error(BB_ERR_ARGUMENT, "sets run past the last bin");
    // the element window and the number of counter replicas follow from
    // nelem alone: windows of at most 16 words (64 elements) of a sample,
    // and as many replicas as fit 64 KiB of counters (32 at most: one per
    // lane)
    const uint32_t P = nelem >= 4 ? (uint32_t)nelem / 4u : 1u;
    const uint32_t ww = P < 16u ? P : 16u;
    ByteGeom g;
    g.src = (const uint8_t *)src;
    g.unit_offset = (const long long *)unit_offset;
    g.counts = (unsigned long long *)counts;
    g.nset = nset;
    g.set_origin = set_origin;
    g.sets_per_bin = sets_per_bin;
    g.nthread = nthread;
    g.nelem = nelem;
    g.lg_p = (uint32_t)__builtin_ctz(P);
    g.lg_ww = (uint32_t)__builtin_ctz(ww);
    g.nwin = P / ww;
    g.ne = nelem >= 4 ? 4u * ww : (uint32_t)nelem;
    g.nrep = 64u / g.ne < 32u ? 64u / g.ne : 32u;
    g.nq = (uint32_t)(payload_nbytes / 4) / P * ww;
    g.nseg = (g.nq + kByteSegQuads * 4u - 1u) / (kByteSegQuads * 4u);
    // three CTAs fit an SM (64 KiB of counters each): two waves, so that the
    // zeroing and read-out of the counters stays small against the payload
    const int64_t items = bp.per_bin * (int64_t)g.nseg;     // per bin
    int64_t split = bp.split_for(6ll * sm_count(), (int64_t)nthread * g.nwin,
                                 items);
    // no CTA reads more than kByteMaxItems segments: its 32-bit counters
    // cannot wrap
    const int64_t need = (items + kByteMaxItems - 1) / kByteMaxItems;
    if (split < need) split = need;
    if (split * g.nwin > 0x7fffffffll || split > 65535)
        return set_error(BB_ERR_UNSUPPORTED,
                         "too many sets or elements for one call");
    g.split = (int)split;
    const size_t smem = (size_t)256 * g.ne * g.nrep * sizeof(uint32_t);
    static bool attr_set = false;
    if (!attr_set) {
        const int rc = check_cuda(cudaFuncSetAttribute(
            k_byte_counts, cudaFuncAttributeMaxDynamicSharedMemorySize,
            kByteCounters * (int)sizeof(uint32_t)), "bb_byte_counts (smem)");
        if (rc != BB_OK) return rc;
        attr_set = true;
    }
    cudaStream_t s = as_stream(stream);
    for (int64_t z0 = 0; z0 < bp.nb; z0 += 65535) {
        const int64_t nz = bp.nb - z0 < 65535 ? bp.nb - z0 : 65535;
        g.bin_first = bp.b0 + z0;
        dim3 grid((unsigned)(split * g.nwin), (unsigned)nthread, (unsigned)nz);
        k_byte_counts<<<grid, kByteBlock, smem, s>>>(g);
        BB_CHECK_LAUNCH("bb_byte_counts");
    }
    return BB_OK;
}


// Mark 4: the (sign, magnitude) states of every channel straight from the
// track words.  Frames are the units (`unit_offset[i]` = offset of frame i's
// payload, i.e. past the 160 header steps, < 0: invalid frame; as written by
// bb_mark4_scan); counts[bin][chan][2 * sign + magnitude].
template <int XF>
static bool m4_field_table(int nchan, int fanout, int ft, int wordbytes,
                           uint8_t (&table)[2][16], std::string &err) {
    uint16_t pos[32];
    int ntrack = 0;
    if (!m4_build_pos(nchan, fanout, ft, pos, ntrack, err)) return false;
    int chan_of[64], mag_of[64];
    for (int b = 0; b < 64; ++b) chan_of[b] = mag_of[b] = -1;
    for (int i = 0; i < nchan * fanout; ++i) {
        chan_of[pos[i] & 0xff] = i % nchan;
        mag_of[pos[i] & 0xff] = 0;
        chan_of[pos[i] >> 8] = i % nchan;
        mag_of[pos[i] >> 8] = 1;
    }
    for (int cls = 0; cls < 2; ++cls)
        for (int f = 0; f < 16; ++f) table[cls][f] = 0xff;
    for (int cls = 0; cls < (wordbytes == 8 ? 2 : 1); ++cls)
        for (int b32 = 0; b32 < 32; ++b32) {
            // a 32-bit load holds half an 8-byte word, one 4-byte word or two
            // 2-byte words of the track stream
            const int b = wordbytes == 8 ? 32 * cls + b32 : b32 % ntrack;
            const uint32_t codes = m4_to_codes<XF>(1u << b32);
            int q = 0;
            while (q < 32 && !((codes >> q) & 1u)) ++q;
            if (q == 32 || (codes & (codes - 1u)) || chan_of[b] < 0
                || (q & 1) != mag_of[b]) {
                err = "internal error: Mark 4 code transform";
                return false;
            }
            const int f = q >> 1;
            if (table[cls][f] != 0xff && table[cls][f] != chan_of[b]) {
                err = "internal error: Mark 4 field table";
                return false;
            }
            table[cls][f] = (uint8_t)chan_of[b];
        }
    return true;
}

extern "C" int bb_mark4_state_counts(
    const void *src, const int64_t *unit_offset, int64_t nframe, int32_t nchan,
    int32_t fanout, int32_t ft, int64_t set_origin, int64_t sets_per_bin,
    uint64_t *counts, int64_t nbin, void *stream) {
    if (!src || !unit_offset || !counts)
        return set_error(BB_ERR_ARGUMENT, "null pointer");
    if (nframe < 0 || set_origin < 0 || sets_per_bin < 1 || nbin < 1)
        return set_error(BB_ERR_ARGUMENT, "bad geometry");
    if (!aligned(src, 4))
        return set_error(BB_ERR_ALIGNMENT, "src must be 4-byte aligned");
    CountGeom g;
    std::string err;
    const int ntrack = nchan * 2 * fanout, wordbytes = ntrack / 8;
    const int xf = ft ? XF_M4_FT : (fanout == 4 && nchan >= 4) ? XF_M4_REORDER
        : XF_M4_NIBBLES;
    const bool ok = xf == XF_M4_FT
        ? m4_field_table<XF_M4_FT>(nchan, fanout, ft, wordbytes, g.field_elem,
                                   err)
        : xf == XF_M4_REORDER
        ? m4_field_table<XF_M4_REORDER>(nchan, fanout, ft, wordbytes,
                                        g.field_elem, err)
        : m4_field_table<XF_M4_NIBBLES>(nchan, fanout, ft, wordbytes,
                                        g.field_elem, err);
    if (!ok) return set_error(BB_ERR_UNSUPPORTED, "%s", err.c_str());
    if (nframe == 0) return BB_OK;
    const int64_t b0 = set_origin / sets_per_bin;
    const int64_t b1 = (set_origin + nframe - 1) / sets_per_bin;
    if (b1 >= nbin)
        return set_error(BB_ERR_ARGUMENT, "frames run past the last bin");
    g.src = (const uint8_t *)src;
    g.unit_offset = (const long long *)unit_offset;
    g.counts = (unsigned long long *)counts;
    g.nset = nframe;
    g.set_origin = set_origin;
    g.sets_per_bin = sets_per_bin;
    g.nthread = 1;
    g.nelem = nchan;
    g.nword = (uint32_t)((20000 - 160) * wordbytes / 4);
    g.nseg = 1u;
    const int P = wordbytes == 8 ? 2 : 1;
    const int64_t nb = b1 - b0 + 1;
    const int64_t per_bin = sets_per_bin < nframe ? sets_per_bin : nframe;
    int64_t split = ((int64_t)count_depth(true) * sm_count() + nb - 1) / nb;
    const int64_t need = (per_bin * (int64_t)g.nword + (1ll << 26) - 1)
        / (1ll << 26);
    const int64_t full = per_bin / (kVertBlock / 32);
    if (split > full) split = full;
    if (split < need) split = need;
    if (split > per_bin) split = per_bin;
    if (split < 1) split = 1;
    if (split > 65535) split = 65535;
    g.split = (int)split;
    const size_t smem = (size_t)3 * 20 * kVertBlock * sizeof(uint32_t);
    cudaStream_t s = as_stream(stream);
    for (int64_t z0 = 0; z0 < nb; z0 += 65535) {
        const int64_t nz = nb - z0 < 65535 ? nb - z0 : 65535;
        g.bin_first = b0 + z0;
        dim3 grid((unsigned)split, 1u, (unsigned)nz);
        if (xf == XF_M4_FT)
            k_state_counts_vert<2, XF_M4_FT><<<grid, kVertBlock, smem, s>>>(g, P);
        else if (xf == XF_M4_REORDER)
            k_state_counts_vert<2, XF_M4_REORDER>
                <<<grid, kVertBlock, smem, s>>>(g, P);
        else
            k_state_counts_vert<2, XF_M4_NIBBLES>
                <<<grid, kVertBlock, smem, s>>>(g, P);
        BB_CHECK_LAUNCH("bb_mark4_state_counts");
    }
    return BB_OK;
}
