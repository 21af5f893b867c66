// Selective decode kernels (subset reads) and their C entry points.
// sm_100a only.  See bb_select.cuh for the layouts and the decomposition.
#include <string>
#include <vector>
#include "bb_runtime.cuh"
#include "bb_select.cuh"

namespace bb {

// One CTA: kSelThreads x kSelGroups output groups, all loads first.  INT8:
// blockIdx.y is the unit, groups count from the unit's first output group.
template <int BPS, int CODEC, bool INT8, typename OT>
__global__ void __launch_bounds__(kSelThreads)
k_decode_select(const SelGeom p, const LevelTable<BPS> lv) {
    using Lut = DecodeLut<BPS>;
    __shared__ __align__(128) float lut[CODEC == CODEC_LEVELS ? Lut::kFloats : 2];
    __shared__ SelEntry tab[kSelSmem];
    if (CODEC == CODEC_LEVELS)
        for (int i = threadIdx.x; i < Lut::kFloats; i += kSelThreads)
            lut[i] = Lut::value(lv.v, i);
    if (p.nsel <= kSelSmem)
        for (uint32_t j = threadIdx.x; j < p.nsel; j += kSelThreads)
            tab[j] = sel_entry<INT8>(p, j);
    __syncthreads();
    long long ue0 = 0, ue1 = 0, g0 = p.g0;
    uint32_t ngroups = p.ngroups;
    const uint32_t unit = blockIdx.y;
    if (INT8) {
        if (p.unit_offset[unit] < 0) return;
        sel_unit_range(p, unit, ue0, ue1);
        g0 = floor4(ue0 + p.head);
        ngroups = (uint32_t)(floor4(ue1 + p.head + 3) - g0);
    }
    const uint32_t k0 = blockIdx.x * (kSelThreads * kSelGroups) + threadIdx.x;
    uint32_t w[kSelGroups][4], meta[kSelGroups][4];
#pragma unroll
    for (int k = 0; k < kSelGroups; ++k) {
        const uint32_t gi = k0 + k * kSelThreads;
        if (gi < ngroups)
            sel_fetch<BPS, INT8>(p, tab, g0 + gi, unit, ue0, ue1, w[k],
                                 meta[k]);
    }
#pragma unroll
    for (int k = 0; k < kSelGroups; ++k) {
        const uint32_t gi = k0 + k * kSelThreads;
        if (gi < ngroups)
            sel_emit<BPS, CODEC, OT>(p, lut, g0 + gi, w[k], meta[k]);
    }
}

inline unsigned sel_grid(uint32_t ngroups) {
    const uint32_t per = kSelThreads * kSelGroups;
    return (ngroups + per - 1) / per;
}

template <int BPS, int CODEC, typename OT>
static int launch_select(const std::vector<SelGeom> &launches,
                         const float *levels_host, cudaStream_t stream) {
    LevelTable<BPS> lv;
    for (int i = 0; i < (1 << BPS); ++i)
        lv.v[i] = (CODEC == CODEC_LEVELS && levels_host) ? levels_host[i] : 0.f;
    for (const SelGeom &g : launches) {
        k_decode_select<BPS, CODEC, false, OT>
            <<<sel_grid(g.ngroups), kSelThreads, 0, stream>>>(g, lv);
        BB_CHECK_LAUNCH("bb_decode_select_bitfield launch");
    }
    return BB_OK;
}

template <typename OT>
static int dispatch_select(int bps, int codec, const float *levels_host,
                           const std::vector<SelGeom> &l, cudaStream_t s) {
    if (codec == BB_CODEC_LEVELS) {
        switch (bps) {
        case 1: return launch_select<1, CODEC_LEVELS, OT>(l, levels_host, s);
        case 2: return launch_select<2, CODEC_LEVELS, OT>(l, levels_host, s);
        case 4: return launch_select<4, CODEC_LEVELS, OT>(l, levels_host, s);
        case 8:
            if (affine8_matches(levels_host))       // the standard 8-bit table
                return launch_select<8, CODEC_AFFINE8, OT>(l, nullptr, s);
            return launch_select<8, CODEC_LEVELS, OT>(l, levels_host, s);
        }
    } else if (codec == BB_CODEC_SINT) {
        switch (bps) {
        case 4: return launch_select<4, CODEC_SINT, OT>(l, nullptr, s);
        case 8: return launch_select<8, CODEC_SINT, OT>(l, nullptr, s);
        }
    }
    return set_error(BB_ERR_UNSUPPORTED, "no decoder for bps=%d codec=%d", bps,
                     codec);
}

template <typename OT>
static void launch_select_int8(const SelGeom &g, uint32_t ngroups_max,
                               int64_t nunit, cudaStream_t s) {
    const LevelTable<8> lv = LevelTable<8>();
    for (int64_t u0 = 0; u0 < nunit; u0 += 65535) {
        SelGeom gu = g;
        const int64_t n = nunit - u0 < 65535 ? nunit - u0 : 65535;
        gu.unit_offset += u0;
        gu.t_begin += u0;
        gu.t_end += u0;
        gu.out_t0 += u0;
        k_decode_select<8, CODEC_SINT, true, OT>
            <<<dim3(sel_grid(ngroups_max), (unsigned)n), kSelThreads, 0, s>>>(
                gu, lv);
    }
}

}  // namespace bb

using namespace bb;

extern "C" int bb_decode_select_bitfield(
    const void *src, const int64_t *unit_offset, int64_t nset, int32_t nthread,
    int64_t payload_nbytes, int32_t bps, int32_t nelem, int32_t complex_data,
    int32_t codec, const float *levels_host, float fill_value,
    int64_t sample_start, int64_t nsample, const int32_t *sel, int32_t nsel,
    int32_t out_dtype, void *out, void *stream) {
    if (!src || !unit_offset || !sel || !out)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    const int esize = out_elem_nbytes(out_dtype);
    if (esize == 0)
        return set_error(BB_ERR_ARGUMENT,
                         "out_dtype must be BB_F32, BB_F16 or BB_BF16");
    if (!aligned(out, esize) || !aligned(src, 4))
        return set_error(BB_ERR_ALIGNMENT,
                         "out must be %d-byte and src 4-byte aligned", esize);
    if (codec == BB_CODEC_LEVELS && !levels_host)
        return set_error(BB_ERR_ARGUMENT, "levels_host required");
    std::vector<SelGeom> launches;
    std::string err;
    if (!plan_select_bitfield(src, unit_offset, nset, nthread, payload_nbytes,
                              bps, nelem, complex_data, fill_value,
                              sample_start, nsample, sel, nsel, out, esize,
                              launches, err))
        return set_error(BB_ERR_ARGUMENT, "%s", err.c_str());
    cudaStream_t s = as_stream(stream);
    if (out_dtype == BB_F16)
        return dispatch_select<F16>(bps, codec, levels_host, launches, s);
    if (out_dtype == BB_BF16)
        return dispatch_select<BF16>(bps, codec, levels_host, launches, s);
    return dispatch_select<float>(bps, codec, levels_host, launches, s);
}

extern "C" int bb_decode_select_int8(
    const void *src, const int64_t *unit_offset, int64_t nunit,
    int64_t nsample, int64_t heap, int64_t heap_stride, int64_t t_stride,
    const int32_t *off, int32_t nsel, const int64_t *t_begin,
    const int64_t *t_end, const int64_t *out_t0, int32_t out_dtype, void *out,
    void *stream) {
    if (!src || !unit_offset || !off || !t_begin || !t_end || !out_t0 || !out)
        return set_error(BB_ERR_ARGUMENT, "null pointer argument");
    const int esize = out_elem_nbytes(out_dtype);
    if (esize == 0)
        return set_error(BB_ERR_ARGUMENT,
                         "out_dtype must be BB_F32, BB_F16 or BB_BF16");
    if (!aligned(out, esize))
        return set_error(BB_ERR_ALIGNMENT, "out must be %d-byte aligned",
                         esize);
    SelGeom g;
    uint32_t ngroups_max;
    std::string err;
    if (!plan_select_int8(src, unit_offset, nunit, nsample, heap, heap_stride,
                          t_stride, off, nsel, t_begin, t_end, out_t0, out,
                          esize, g, ngroups_max, err))
        return set_error(BB_ERR_ARGUMENT, "%s", err.c_str());
    if (nunit == 0 || nsample == 0) return BB_OK;
    cudaStream_t s = as_stream(stream);
    if (out_dtype == BB_F16) launch_select_int8<F16>(g, ngroups_max, nunit, s);
    else if (out_dtype == BB_BF16)
        launch_select_int8<BF16>(g, ngroups_max, nunit, s);
    else launch_select_int8<float>(g, ngroups_max, nunit, s);
    BB_CHECK_LAUNCH("bb_decode_select_int8 launch");
    return BB_OK;
}
