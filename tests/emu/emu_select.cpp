// CPU emulation of the selective decoders — TEST INFRASTRUCTURE ONLY.
// The same planning and per-thread bodies as csrc/bb_select.cu; every CTA's
// table and level fill, then its threads' fetch and emit phases, run as loops.
#include <string>
#include <vector>
#include "../../baseband_b200/csrc/bb_select.cuh"
#include "../../include/baseband_b200.h"

using namespace bb;

namespace {

int esize_of(int32_t out_dtype) {
    return out_dtype == BB_F32 ? 4
        : (out_dtype == BB_F16 || out_dtype == BB_BF16) ? 2 : 0;
}

template <int BPS, int CODEC, bool INT8, typename OT>
void run_cta(const SelGeom &p, const float *levels, uint32_t block,
             uint32_t unit) {
    using Lut = DecodeLut<BPS>;
    std::vector<float> lut(Lut::kFloats);
    if (CODEC == CODEC_LEVELS)
        for (int i = 0; i < Lut::kFloats; ++i) lut[i] = Lut::value(levels, i);
    std::vector<SelEntry> tab(kSelSmem);
    if (p.nsel <= kSelSmem)
        for (uint32_t j = 0; j < p.nsel; ++j) tab[j] = sel_entry<INT8>(p, j);
    long long ue0 = 0, ue1 = 0, g0 = p.g0;
    uint32_t ngroups = p.ngroups;
    if (INT8) {
        if (p.unit_offset[unit] < 0) return;
        sel_unit_range(p, unit, ue0, ue1);
        g0 = floor4(ue0 + p.head);
        ngroups = (uint32_t)(floor4(ue1 + p.head + 3) - g0);
    }
    for (uint32_t t = 0; t < (uint32_t)kSelThreads; ++t) {
        const uint32_t k0 = block * (kSelThreads * kSelGroups) + t;
        uint32_t w[kSelGroups][4], meta[kSelGroups][4];
        for (int k = 0; k < kSelGroups; ++k) {
            const uint32_t gi = k0 + k * kSelThreads;
            if (gi < ngroups)
                sel_fetch<BPS, INT8>(p, tab.data(), g0 + gi, unit, ue0, ue1,
                                     w[k], meta[k]);
        }
        for (int k = 0; k < kSelGroups; ++k) {
            const uint32_t gi = k0 + k * kSelThreads;
            if (gi < ngroups)
                sel_emit<BPS, CODEC, OT>(p, lut.data(), g0 + gi, w[k],
                                         meta[k]);
        }
    }
}

uint32_t nblocks(uint32_t ngroups) {
    const uint32_t per = kSelThreads * kSelGroups;
    return (ngroups + per - 1) / per;
}

template <int BPS, int CODEC, typename OT>
int run_bitfield(const std::vector<SelGeom> &launches, const float *levels) {
    float lv[256] = {0.f};
    for (int i = 0; i < (1 << BPS); ++i)
        lv[i] = (CODEC == CODEC_LEVELS && levels) ? levels[i] : 0.f;
    for (const SelGeom &g : launches)
        for (uint32_t b = 0; b < nblocks(g.ngroups); ++b)
            run_cta<BPS, CODEC, false, OT>(g, lv, b, 0);
    return 0;
}

template <typename OT>
int dispatch(int bps, int codec, const float *levels,
             const std::vector<SelGeom> &l) {
    if (codec == BB_CODEC_LEVELS) {
        switch (bps) {
        case 1: return run_bitfield<1, CODEC_LEVELS, OT>(l, levels);
        case 2: return run_bitfield<2, CODEC_LEVELS, OT>(l, levels);
        case 4: return run_bitfield<4, CODEC_LEVELS, OT>(l, levels);
        case 8:
            if (affine8_matches(levels))
                return run_bitfield<8, CODEC_AFFINE8, OT>(l, nullptr);
            return run_bitfield<8, CODEC_LEVELS, OT>(l, levels);
        }
    } else if (codec == BB_CODEC_SINT) {
        switch (bps) {
        case 4: return run_bitfield<4, CODEC_SINT, OT>(l, nullptr);
        case 8: return run_bitfield<8, CODEC_SINT, OT>(l, nullptr);
        }
    }
    return BB_ERR_UNSUPPORTED;
}

template <typename OT>
void run_int8(const SelGeom &g, uint32_t ngroups_max, int64_t nunit) {
    for (int64_t u = 0; u < nunit; ++u)
        for (uint32_t b = 0; b < nblocks(ngroups_max); ++b)
            run_cta<8, CODEC_SINT, true, OT>(g, nullptr, b, (uint32_t)u);
}

}  // namespace

extern "C" {

int bb_decode_select_bitfield(
    const void *src, const int64_t *unit_offset, int64_t nset, int32_t nthread,
    int64_t payload_nbytes, int32_t bps, int32_t nelem, int32_t complex_data,
    int32_t codec, const float *levels_host, float fill_value,
    int64_t sample_start, int64_t nsample, const int32_t *sel, int32_t nsel,
    int32_t out_dtype, void *out, void *stream) {
    const int esize = esize_of(out_dtype);
    if (!src || !unit_offset || !sel || !out || esize == 0)
        return BB_ERR_ARGUMENT;
    if (((uintptr_t)out % esize) || ((uintptr_t)src % 4))
        return BB_ERR_ALIGNMENT;
    if (codec == BB_CODEC_LEVELS && !levels_host) return BB_ERR_ARGUMENT;
    std::vector<SelGeom> launches;
    std::string err;
    if (!plan_select_bitfield(src, unit_offset, nset, nthread, payload_nbytes,
                              bps, nelem, complex_data, fill_value,
                              sample_start, nsample, sel, nsel, out, esize,
                              launches, err))
        return BB_ERR_ARGUMENT;
    if (out_dtype == BB_F16)
        return dispatch<F16>(bps, codec, levels_host, launches);
    if (out_dtype == BB_BF16)
        return dispatch<BF16>(bps, codec, levels_host, launches);
    return dispatch<float>(bps, codec, levels_host, launches);
}

int bb_decode_select_int8(
    const void *src, const int64_t *unit_offset, int64_t nunit,
    int64_t nsample, int64_t heap, int64_t heap_stride, int64_t t_stride,
    const int32_t *off, int32_t nsel, const int64_t *t_begin,
    const int64_t *t_end, const int64_t *out_t0, int32_t out_dtype, void *out,
    void *stream) {
    const int esize = esize_of(out_dtype);
    if (!src || !unit_offset || !off || !t_begin || !t_end || !out_t0 || !out
        || esize == 0)
        return BB_ERR_ARGUMENT;
    if ((uintptr_t)out % esize) return BB_ERR_ALIGNMENT;
    SelGeom g;
    uint32_t ngroups_max;
    std::string err;
    if (!plan_select_int8(src, unit_offset, nunit, nsample, heap, heap_stride,
                          t_stride, off, nsel, t_begin, t_end, out_t0, out,
                          esize, g, ngroups_max, err))
        return BB_ERR_ARGUMENT;
    if (nunit == 0 || nsample == 0) return 0;
    if (out_dtype == BB_F16) run_int8<F16>(g, ngroups_max, nunit);
    else if (out_dtype == BB_BF16) run_int8<BF16>(g, ngroups_max, nunit);
    else run_int8<float>(g, ngroups_max, nunit);
    return 0;
}

}  // extern "C"
