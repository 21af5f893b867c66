// Shared helpers for the baseband_b200 kernels.
//
// The per-thread bodies of the streaming kernels are written as
// host/device inline functions over plain structs so that the index
// arithmetic can also be compiled by g++ for the CPU emulation used by
// tests/test_emulation.py (test infrastructure; the shipped library only
// contains the CUDA instantiations).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define BB_HD __host__ __device__ __forceinline__
#else
#define BB_HD inline
#endif

namespace bb {

struct alignas(16) F4 { float x, y, z, w; };
struct alignas(16) D2 { double x, y; };
struct alignas(8) F2 { float x, y; };
struct alignas(16) U4 { uint32_t x, y, z, w; };

BB_HD uint32_t umulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

// PRMT: byte i of the result is byte (s >> 4i) & 7 of the pair {x, y}
// (selector nibbles 0..7 only: no sign replication).
BB_HD uint32_t byte_perm(uint32_t x, uint32_t y, uint32_t s) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, y, s);
#else
    const uint64_t xy = ((uint64_t)y << 32) | x;
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i)
        r |= (uint32_t)((xy >> (8 * ((s >> (4 * i)) & 7u))) & 0xffu) << (8 * i);
    return r;
#endif
}

// Division of any 32-bit unsigned n by a runtime-constant d >= 1
// (Granlund & Montgomery round-up method): 4 integer instructions.
struct FastDiv {
    uint32_t d, mul, sh1, sh2;
    BB_HD uint32_t div(uint32_t n) const {
        uint32_t t = umulhi32(mul, n);
        return (t + ((n - t) >> sh1)) >> sh2;
    }
    BB_HD void divmod(uint32_t n, uint32_t &q, uint32_t &r) const {
        q = div(n);
        r = n - q * d;
    }
};

inline FastDiv make_fastdiv(uint32_t d) {
    FastDiv f;
    f.d = d;
    uint32_t l = 0;
    while ((1ull << l) < d) ++l;                 // ceil(log2 d)
    f.mul = (uint32_t)((((1ull << l) - d) << 32) / d + 1);
    f.sh1 = l < 1 ? l : 1;
    f.sh2 = l > 1 ? l - 1 : 0;
    return f;
}

inline int ilog2_exact(uint32_t v) {            // -1 if not a power of two
    if (v == 0 || (v & (v - 1))) return -1;
    int l = 0;
    while ((1u << l) < v) ++l;
    return l;
}

// Arithmetic that must round exactly once per numpy ufunc (no FMA fusion).
BB_HD float add_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    volatile float r = a + b; return r;
#endif
}
BB_HD float mul_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    volatile float r = a * b; return r;
#endif
}
// Fused multiply-add, one rounding (explicitly wanted: not an accidental
// contraction, which the build disables with -fmad=false).
BB_HD float fma_rn(float a, float b, float c) {
#if defined(__CUDA_ARCH__)
    return __fmaf_rn(a, b, c);
#else
    return __builtin_fmaf(a, b, c);
#endif
}
BB_HD float uint_as_float(uint32_t u) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f;
    __builtin_memcpy(&f, &u, 4);
    return f;
#endif
}
// Small signed integer (|i| < 2^22) -> float without the conversion pipe: i is
// added to the mantissa of 1.5 * 2^23, whose ulp is 1, and the offset removed
// by one exact subtraction.
BB_HD float small_int_to_float(int32_t i) {
    return add_rn(uint_as_float(0x4B400000u + (uint32_t)i), -12582912.0f);
}
// ------------------------------------------------- decoder output element types
// A decoder writes float32 (`float`) or the 16-bit patterns of IEEE half
// (F16) or bfloat16 (BF16).  The kernels compute every value in float32 and
// round it to the output type once, when it is stored (round to nearest even,
// overflow to +-inf: torch's `.to(dtype)`), so a reduced-precision result is
// the float32 result converted elementwise.
struct alignas(2) F16 { uint16_t bits; static constexpr bool kBrain = false; };
struct alignas(2) BF16 { uint16_t bits; static constexpr bool kBrain = true; };
struct alignas(8) H4 { uint32_t lo, hi; };

BB_HD uint32_t float_as_uint(float f) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(f);
#else
    uint32_t u;
    __builtin_memcpy(&u, &f, 4);
    return u;
#endif
}

// Host rounding of a float32 bit pattern (the CPU emulation and the tests).
// NaN keeps its sign and becomes a quiet NaN; its payload is not specified.
inline uint16_t f32_to_f16_bits(uint32_t x) {
    const uint32_t sign = (x >> 16) & 0x8000u, ax = x & 0x7fffffffu;
    if (ax > 0x7f800000u) return (uint16_t)(sign | 0x7e00u);
    if (ax >= 0x477ff000u) return (uint16_t)(sign | 0x7c00u);  // >= 65520
    if (ax >= 0x38800000u) {                                 // normal half
        const uint32_t r = ax + 0xfffu + ((ax >> 13) & 1u);
        return (uint16_t)(sign | ((r >> 13) - 0x1c000u));
    }
    const uint32_t e = ax >> 23;                             // subnormal half
    if (e < 102) return (uint16_t)sign;                      // < 2^-25
    const uint32_t m = (ax & 0x7fffffu) | 0x800000u, s = 126 - e;
    uint32_t q = m >> s;
    const uint32_t rem = m & ((1u << s) - 1u), half = 1u << (s - 1);
    if (rem > half || (rem == half && (q & 1u))) ++q;
    return (uint16_t)(sign | q);
}

inline uint16_t f32_to_bf16_bits(uint32_t x) {
    if ((x & 0x7fffffffu) > 0x7f800000u)
        return (uint16_t)(((x >> 16) & 0x8000u) | 0x7fc0u);
    return (uint16_t)((x + 0x7fffu + ((x >> 16) & 1u)) >> 16);
}

// Two float32 -> two values of OT (F16 / BF16) in one word, `lo` in the low
// half: one cvt.rn.{f16,bf16}x2.f32 on the device.
template <typename OT>
BB_HD uint32_t pack_half2(float lo, float hi) {
#if defined(__CUDA_ARCH__)
    uint32_t r;
    if (OT::kBrain)
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    else
        asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
#else
    const uint32_t a = float_as_uint(lo), b = float_as_uint(hi);
    if (OT::kBrain)
        return f32_to_bf16_bits(a) | ((uint32_t)f32_to_bf16_bits(b) << 16);
    return f32_to_f16_bits(a) | ((uint32_t)f32_to_f16_bits(b) << 16);
#endif
}

// Stores of 4, 2 and 1 decoded values at an element pointer of the output
// type: 16/8/4 bytes for float32, 8/4/2 for the 16-bit types.
BB_HD void store4(float *p, const F4 &v) { *reinterpret_cast<F4 *>(p) = v; }
BB_HD void store2(float *p, const F2 &v) { *reinterpret_cast<F2 *>(p) = v; }
BB_HD void store1(float *p, float v) { *p = v; }
template <typename OT>
BB_HD void store4(OT *p, const F4 &v) {
    *reinterpret_cast<H4 *>(p) = H4{pack_half2<OT>(v.x, v.y),
                                    pack_half2<OT>(v.z, v.w)};
}
template <typename OT>
BB_HD void store2(OT *p, const F2 &v) {
    *reinterpret_cast<uint32_t *>(p) = pack_half2<OT>(v.x, v.y);
}
template <typename OT>
BB_HD void store1(OT *p, float v) {
    p->bits = (uint16_t)pack_half2<OT>(v, 0.f);
}

// The output of a geometry struct (`void *out`) as elements of OT.
template <typename OT, typename Geom>
BB_HD OT *out_as(const Geom &p) { return static_cast<OT *>(p.out); }

// -------------------------------------------------- encoder input element types
// An encoder reads its input as the storage type S (float, double, F16, BF16)
// and quantises in the arithmetic type arith_t<S>: double for double, float
// for the rest.  A 16-bit value is widened to float32 once, as it is loaded;
// widening is exact, so it encodes to the bits its float32 value would.
template <typename S> struct Arith { using type = S; };
template <> struct Arith<F16> { using type = float; };
template <> struct Arith<BF16> { using type = float; };
template <typename S> using arith_t = typename Arith<S>::type;

// Host widening of a half bit pattern (the CPU emulation): exact for every
// value, NaN keeps its sign and payload.
inline uint32_t f16_to_f32_bits(uint32_t h) {
    const uint32_t sign = (h & 0x8000u) << 16;
    uint32_t e = (h >> 10) & 0x1fu, m = h & 0x3ffu;
    if (e == 0x1fu) return sign | 0x7f800000u | (m << 13);  // inf / NaN
    if (e == 0) {
        if (m == 0) return sign;                              // +-0
        e = 1;                                                // subnormal
        while (!(m & 0x400u)) { m <<= 1; --e; }
        m &= 0x3ffu;
    }
    return sign | ((e + 112u) << 23) | (m << 13);
}

// The two 16-bit values of S in one word (`lo` from the low half) -> float32.
// bfloat16 is the high half of a float32: a shift and a mask.  Half takes one
// cvt.f32.f16 each; a NaN's sign is then put back from the input, since only
// the sign of a NaN can reach a code (the Mark 5B 1-bit quantiser).
template <typename S>
BB_HD void widen_half2(uint32_t u, float &lo, float &hi) {
    if (S::kBrain) {
        lo = uint_as_float(u << 16);
        hi = uint_as_float(u & 0xffff0000u);
        return;
    }
#if defined(__CUDA_ARCH__)
    asm("{.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\t"
        "cvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;}"
        : "=f"(lo), "=f"(hi) : "r"(u));
    lo = uint_as_float(float_as_uint(lo) | ((u << 16) & 0x80000000u));
    hi = uint_as_float(float_as_uint(hi) | (u & 0x80000000u));
#else
    lo = uint_as_float(f16_to_f32_bits(u & 0xffffu));
    hi = uint_as_float(f16_to_f32_bits(u >> 16));
#endif
}

// One input value in the arithmetic type.
BB_HD float widen(float x) { return x; }
BB_HD double widen(double x) { return x; }
template <typename S>
BB_HD float widen(S x) {
    float lo, hi;
    widen_half2<S>(x.bits, lo, hi);
    return lo;
}

// Four consecutive input values from one vector load: 16 bytes for float32,
// two 16-byte loads for float64, 8 bytes for the 16-bit types.
BB_HD void load4(const float *p, float v[4]) {
    const F4 r = *reinterpret_cast<const F4 *>(p);
    v[0] = r.x; v[1] = r.y; v[2] = r.z; v[3] = r.w;
}
BB_HD void load4(const double *p, double v[4]) {
    const D2 a = reinterpret_cast<const D2 *>(p)[0];
    const D2 b = reinterpret_cast<const D2 *>(p)[1];
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
template <typename S>
BB_HD void load4(const S *p, float v[4]) {
    const H4 h = *reinterpret_cast<const H4 *>(p);
    widen_half2<S>(h.lo, v[0], v[1]);
    widen_half2<S>(h.hi, v[2], v[3]);
}

BB_HD double add_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    volatile double r = a + b; return r;
#endif
}
BB_HD double mul_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    volatile double r = a * b; return r;
#endif
}

}  // namespace bb
