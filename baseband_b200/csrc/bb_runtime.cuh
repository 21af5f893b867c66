// Host-side runtime helpers shared by the launchers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/baseband_b200.h"

namespace bb {

int set_error(int code, const char *fmt, ...);
int check_cuda(cudaError_t err, const char *what);
int sm_count();                       // of the current device (cached)

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

// Grid for a grid-stride streaming kernel: enough CTAs of `block` threads to
// fill every SM `ctas_per_sm` deep, never more than the work needs.
int grid_override();                  // BB_CTAS_PER_SM (tuning): -1 unset, 0 = full

inline unsigned stream_grid(uint64_t nitems, unsigned block, unsigned ctas_per_sm) {
    uint64_t need = (nitems + block - 1) / block;
    int ov = grid_override();
    if (ov == 0) return (unsigned)(need ? need : 1);
    if (ov > 0) ctas_per_sm = (unsigned)ov;
    uint64_t cap = (uint64_t)sm_count() * ctas_per_sm;
    uint64_t g = need < cap ? need : cap;
    return (unsigned)(g ? g : 1);
}

inline bool aligned(const void *p, uintptr_t a) {
    return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0;
}

// Bytes per element of a decoder output type (bb_dtype), 0 if a decoder
// cannot write it.
inline int out_elem_nbytes(int32_t out_dtype) {
    return out_dtype == BB_F32 ? 4
        : (out_dtype == BB_F16 || out_dtype == BB_BF16) ? 2 : 0;
}

// Alignment an encoder requires of its input (one vector load of four
// values: 16 bytes for float32 and float64, 8 for the 16-bit types), 0 if an
// encoder cannot read the type.
inline int in_vec_align(int32_t in_dtype) {
    return (in_dtype == BB_F32 || in_dtype == BB_F64) ? 16
        : (in_dtype == BB_F16 || in_dtype == BB_BF16) ? 8 : 0;
}

#define BB_CHECK_LAUNCH(what)                                            \
    do {                                                                 \
        cudaError_t e__ = cudaGetLastError();                            \
        if (e__ != cudaSuccess) return bb::check_cuda(e__, what);        \
    } while (0)

}  // namespace bb
