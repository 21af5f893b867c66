/*
 * baseband_b200 — C ABI of the B200 (sm_100a) sample codec library.
 *
 * This is the drop-in boundary for the data-parallel hot path of
 * mhvk/baseband (reference paths below are relative to the reference
 * checkout, `file:line`).  The reference is pure Python + numpy; each entry
 * point replaces one family of numpy ufunc chains and is what a ctypes
 * binding inside the reference's `_decoders` / `_encoders` tables, `Frame`
 * classes and `StreamReaderBase.read` / `StreamWriterBase.write` would call
 * (see INTEGRATION.md for the reference-side stubs).
 *
 * Conventions
 *  - plain C types only; every buffer is caller-owned; the library never
 *    allocates result memory and keeps no state besides the last error text.
 *  - `src`, `dst`, `out`, `in`, `unit_offset`, `valid` ... are DEVICE
 *    pointers unless the name ends in `_host`.
 *  - `stream` is a `cudaStream_t` passed as `void*` (NULL = default stream).
 *    All work is stream-ordered; nothing synchronises the host.
 *  - return value: BB_OK or a negative bb_status; `bb_last_error()` gives a
 *    thread-local text.  No exceptions cross this boundary.
 *  - "unit" = the payload of one frame (VDIF: one thread-frame).  A decode
 *    call is handed a table `unit_offset[nset * nthread]` of byte offsets of
 *    each payload inside `src`; a negative offset marks an invalid or missing
 *    frame whose samples are replaced by `fill_value`
 *    (baseband/base/frame.py:191-199).
 *  - sample order and bit layouts are those of SURVEY.md appendix A; results
 *    are bit-identical to the reference numpy path.
 */
#ifndef BASEBAND_B200_H
#define BASEBAND_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BB_ABI_VERSION 2

typedef enum bb_status {
    BB_OK = 0,
    BB_ERR_ARGUMENT = -1,     /* bad size / combination (ValueError upstream) */
    BB_ERR_ALIGNMENT = -2,    /* pointer or offset not aligned as required */
    BB_ERR_UNSUPPORTED = -3,  /* no such codec (KeyError upstream) */
    BB_ERR_CUDA = -4          /* CUDA runtime error, see bb_last_error() */
} bb_status;

/* Code -> value rule for the generic bit-field codec. */
typedef enum bb_codec {
    BB_CODEC_LEVELS = 0,  /* value = levels[code]; VDIF offset binary
                             (baseband/vdif/payload.py:25-103), Mark 5B
                             sign/magnitude (baseband/mark5b/payload.py:27-94),
                             VDIF 8 bit (baseband/base/encoding.py:131-144) */
    BB_CODEC_SINT = 1     /* value = two's complement integer of the code;
                             GSB nibbles (baseband/gsb/payload.py:24-42),
                             DADA/GUPPI/GSB int8 (dada/payload.py:13-14) */
} bb_codec;

/* Quantiser family for encoding. */
typedef enum bb_quantiser {
    BB_QUANT_OFFSET_BINARY = 0, /* baseband/base/encoding.py:63-128,147-158
                                   packed LSB first, vdif/payload.py:77-114 */
    BB_QUANT_MARK5B = 1,        /* 1 bit = signbit, 2 bit codes 1<->2 swapped
                                   (baseband/mark5b/payload.py:86-106) */
    BB_QUANT_SINT = 2           /* clip(rint(v)) two's complement; 4 and 8 bit
                                   (gsb/payload.py:45-53, guppi/payload.py:17) */
} bb_quantiser;

/* Element types.  Encoders take BB_F32 / BB_F64 input or, through the
 * `_typed` entry points, BB_F16 (IEEE half) / BB_BF16 (bfloat16); a 16-bit
 * input value encodes to exactly the bits of its float32 value (widening is
 * exact).  Decoders write BB_F32 or, through the `_typed` entry points,
 * BB_F16 / BB_BF16.  A 16-bit result is the float32 result rounded
 * elementwise to nearest even (overflow to +-inf), as torch's `.to(dtype)`
 * converts it. */
typedef enum bb_dtype {
    BB_F32 = 0, BB_F64 = 1, BB_F16 = 2, BB_BF16 = 3
} bb_dtype;

/* ---------------------------------------------------------------- runtime */
int bb_abi_version(void);
const char *bb_last_error(void);
int bb_device_count(void);
int bb_set_device(int device);
int bb_device_sm_count(int device);
/* Raw memory/stream helpers so that a host without torch can drive the
 * library (the Python layer uses torch allocations and these copies). */
int bb_malloc(void **ptr, int64_t nbytes);
int bb_free(void *ptr);
int bb_host_alloc(void **ptr_host, int64_t nbytes);      /* pinned */
int bb_host_free(void *ptr_host);
int bb_host_register(void *ptr_host, int64_t nbytes);    /* pin in place */
int bb_host_unregister(void *ptr_host);
int bb_memcpy_h2d(void *dst, const void *src_host, int64_t nbytes, void *stream);
int bb_memcpy_d2h(void *dst_host, const void *src, int64_t nbytes, void *stream);
int bb_memset(void *dst, int value, int64_t nbytes, void *stream);
int bb_stream_create(void **stream);
int bb_stream_destroy(void *stream);
int bb_stream_synchronize(void *stream);

/* ------------------------------------------------- generic bit-field codec
 * Replaces: VDIF `decode_1bit/2bit/4bit` (baseband/vdif/payload.py:69-103),
 * `decode_8bit` (baseband/base/encoding.py:131-144), Mark 5B
 * `decode_1bit/2bit` (baseband/mark5b/payload.py:78-94), GSB
 * `decode_4bit/8bit` (baseband/gsb/payload.py:24-42), DADA `decode_8bit`
 * (baseband/dada/payload.py:13-14), the `.view(dtype).reshape` of
 * `PayloadBase._decode/__getitem__` (baseband/base/payload.py:314-330), the
 * per-frame validity fill (baseband/base/frame.py:191-199) and the thread
 * interleave of `VDIFFrameSet.__getitem__` (baseband/vdif/frame.py:402-434),
 * batched over all frames a `StreamReaderBase.read` call touches
 * (baseband/base/base.py:919-969).
 *
 * Layout: a unit holds `payload_nbytes` bytes = codes of `bps` bits, LSB
 * first, in order [time][nelem]; nelem = nchan * (2 if complex).
 * out[(set*spf + t - sample_start) * nthread * nelem + slot * nelem + e]
 *   for rows 0 <= set*spf + t - sample_start < nsample,
 * spf = payload_nbytes*8 / (bps*nelem).  complex_data only affects the fill
 * (fill_value + 0j).  levels_host: 2^bps floats (BB_CODEC_LEVELS), ignored
 * for BB_CODEC_SINT.  Requirements: payload offsets and payload_nbytes
 * multiples of 4; out 16-byte aligned.
 */
int bb_decode_bitfield(const void *src, const int64_t *unit_offset,
                       int64_t nset, int32_t nthread, int64_t payload_nbytes,
                       int32_t bps, int32_t nelem, int32_t complex_data,
                       int32_t codec, const float *levels_host,
                       float fill_value, int64_t sample_start,
                       int64_t nsample, float *out, void *stream);
/* The same with the output element type chosen by `out_dtype`: BB_F32 (the
 * call above, out 16-byte aligned), BB_F16 or BB_BF16 (out 8-byte aligned;
 * each value is the float32 result rounded to nearest even).  The work
 * decomposition is the same for every output type. */
int bb_decode_bitfield_typed(const void *src, const int64_t *unit_offset,
                             int64_t nset, int32_t nthread,
                             int64_t payload_nbytes, int32_t bps,
                             int32_t nelem, int32_t complex_data,
                             int32_t codec, const float *levels_host,
                             float fill_value, int64_t sample_start,
                             int64_t nsample, int32_t out_dtype, void *out,
                             void *stream);

/* Inverse: quantise + pack `in` (same logical layout as `out` above, float32
 * or float64 — arithmetic is done in the input width exactly as numpy does,
 * baseband/base/encoding.py:63-128) into the payload of every unit with a
 * non-negative offset.  Whole frames only (sample_start = 0, nsample =
 * nset*spf).  Replaces `encode_*` (baseband/vdif/payload.py:77-114,
 * baseband/mark5b/payload.py:86-106, baseband/gsb/payload.py:45-53),
 * `PayloadBase._encode/__setitem__` (baseband/base/payload.py:317-348),
 * `VDIFFrameSet.fromdata` thread split (baseband/vdif/frame.py:288-289) and
 * the per-frame loop of `StreamWriterBase.write`
 * (baseband/base/base.py:1276-1308). */
int bb_encode_bitfield(const void *in, int32_t in_dtype, void *dst,
                       const int64_t *unit_offset, int64_t nset,
                       int32_t nthread, int64_t payload_nbytes, int32_t bps,
                       int32_t nelem, int32_t quantiser, void *stream);
/* The same with 16-bit input as well: `in_dtype` BB_F32 / BB_F64 (in 16-byte
 * aligned) or BB_F16 / BB_BF16 (in 8-byte aligned).  Each value is widened
 * to float32 as it is loaded and quantised as float32 input is; the work
 * decomposition is the same for every input type.  The plain function
 * refuses BB_F16 / BB_BF16. */
int bb_encode_bitfield_typed(const void *in, int32_t in_dtype, void *dst,
                             const int64_t *unit_offset, int64_t nset,
                             int32_t nthread, int64_t payload_nbytes,
                             int32_t bps, int32_t nelem, int32_t quantiser,
                             void *stream);

/* ------------------------------------------------------------------ Mark 4
 * Replaces `reorder32/64/64_Ft` + the five `decode_*`/`encode_*` functions
 * (baseband/mark4/payload.py:48-69, :122-300), keyed like
 * `Mark4Payload._decoders` (baseband/mark4/payload.py:333-342) by
 * (nchan, fanout, ft) with ntrack = nchan*2*fanout, plus the
 * header-overwritten-sample fill of `Mark4Frame.__getitem__`
 * (baseband/mark4/frame.py:239-263): each frame contributes
 * spf = 20000*fanout rows of which the first 160*fanout are fill_value.
 * unit_offset[frame] = byte offset of the payload (frame start + ntrack*20),
 * negative = invalid frame (all fill).  levels_host: 4 floats indexed
 * 2*sign+magnitude.  out[(frame*spf + t - sample_start)*nchan + c]. */
int bb_mark4_decode(const void *src, const int64_t *unit_offset,
                    int64_t nframe, int32_t nchan, int32_t fanout, int32_t ft,
                    const float *levels_host, float fill_value,
                    int64_t sample_start, int64_t nsample, float *out,
                    void *stream);
/* Typed output as bb_decode_bitfield_typed (BB_F16 / BB_BF16: out 8-byte
 * aligned). */
int bb_mark4_decode_typed(const void *src, const int64_t *unit_offset,
                          int64_t nframe, int32_t nchan, int32_t fanout,
                          int32_t ft, const float *levels_host,
                          float fill_value, int64_t sample_start,
                          int64_t nsample, int32_t out_dtype, void *out,
                          void *stream);
/* Inverse for whole frames; rows falling in the header region are ignored. */
int bb_mark4_encode(const void *in, int32_t in_dtype, void *dst,
                    const int64_t *unit_offset, int64_t nframe, int32_t nchan,
                    int32_t fanout, int32_t ft, void *stream);
/* 16-bit input as bb_encode_bitfield_typed (BB_F16 / BB_BF16: in 8-byte
 * aligned). */
int bb_mark4_encode_typed(const void *in, int32_t in_dtype, void *dst,
                          const int64_t *unit_offset, int64_t nframe,
                          int32_t nchan, int32_t fanout, int32_t ft,
                          void *stream);
/* Payload-only variants (Mark4Payload.data / .fromdata): nword track words,
 * no header region.  words/out are device pointers. */
int bb_mark4_decode_words(const void *words, int64_t nword, int32_t nchan,
                          int32_t fanout, int32_t ft, const float *levels_host,
                          float *out, void *stream);
int bb_mark4_encode_words(const void *in, int32_t in_dtype, void *words,
                          int64_t nword, int32_t nchan, int32_t fanout,
                          int32_t ft, void *stream);

/* -------------------------------------------- int8 with an axis transpose
 * GUPPI channels-first payloads (baseband/guppi/payload.py:90-110): stored
 * [chan][time][pol][re,im], decoded (time, pol, chan); and MKBF heaps
 * (baseband/dada/payload.py:54-89).  Both are a batched 2-D transpose of
 * `item_nbytes`-byte items (1 = real, 2 = complex) with int8 -> float32:
 *   in  unit u: [nrow][ncol] items        (ncol fastest)
 *   out unit u: [ncol_take][nrow] items   (nrow fastest)
 * Output position of (unit u, column j): row-of-output =
 *   out_col0[u] + j for j in [col_begin[u], col_end[u]) — this expresses the
 * GUPPI overlap rule (baseband/guppi/base.py:203-206, :270-278;
 * baseband/base/base.py:957-967): later frames skip their first `overlap`
 * samples.  All three tables are device int64[nunit]; out_col0 counts output
 * columns (= items of nrow) from `out`. */
int bb_decode_int8_transposed(const void *src, const int64_t *unit_offset,
                              int64_t nunit, int64_t nrow, int64_t ncol,
                              int32_t item_nbytes, const int64_t *col_begin,
                              const int64_t *col_end, const int64_t *out_col0,
                              float *out, void *stream);
/* Typed output (out 8-byte aligned for every type). */
int bb_decode_int8_transposed_typed(const void *src,
                                    const int64_t *unit_offset, int64_t nunit,
                                    int64_t nrow, int64_t ncol,
                                    int32_t item_nbytes,
                                    const int64_t *col_begin,
                                    const int64_t *col_end,
                                    const int64_t *out_col0,
                                    int32_t out_dtype, void *out,
                                    void *stream);
int bb_encode_int8_transposed(const void *in, int32_t in_dtype, void *dst,
                              const int64_t *unit_offset, int64_t nunit,
                              int64_t nrow, int64_t ncol, int32_t item_nbytes,
                              void *stream);
/* 16-bit input as bb_encode_bitfield_typed.  Like the plain function it
 * takes any element-aligned `in`; the fast tile path needs 16-byte (BB_F32,
 * BB_F64) or 8-byte (BB_F16, BB_BF16) alignment. */
int bb_encode_int8_transposed_typed(const void *in, int32_t in_dtype,
                                    void *dst, const int64_t *unit_offset,
                                    int64_t nunit, int64_t nrow, int64_t ncol,
                                    int32_t item_nbytes, void *stream);

/* Time-first GUPPI payloads (PKTFMT other than '1SFA';
 * baseband/guppi/payload.py:97-102 decode, :131-134 encode): unit u at
 * src + unit_offset[u] holds [nsample][nchan][npol] items of item_nbytes
 * int8; samples [t_begin[u], t_end[u]) are written as float32
 * [npol][nchan][item] starting at output sample out_t0[u] (the same window
 * tables as above, counted in samples).  Encode takes whole units,
 * in = [nunit * nsample][npol][nchan][item] float32/float64. */
int bb_decode_int8_timefirst(const void *src, const int64_t *unit_offset,
                             int64_t nunit, int64_t nsample, int32_t nchan,
                             int32_t npol, int32_t item_nbytes,
                             const int64_t *t_begin, const int64_t *t_end,
                             const int64_t *out_t0, float *out, void *stream);
/* Typed output (BB_F32: out 4-byte aligned; BB_F16 / BB_BF16: 8-byte). */
int bb_decode_int8_timefirst_typed(const void *src,
                                   const int64_t *unit_offset, int64_t nunit,
                                   int64_t nsample, int32_t nchan,
                                   int32_t npol, int32_t item_nbytes,
                                   const int64_t *t_begin,
                                   const int64_t *t_end,
                                   const int64_t *out_t0, int32_t out_dtype,
                                   void *out, void *stream);
int bb_encode_int8_timefirst(const void *in, int32_t in_dtype, void *dst,
                             const int64_t *unit_offset, int64_t nunit,
                             int64_t nsample, int32_t nchan, int32_t npol,
                             int32_t item_nbytes, void *stream);
/* 16-bit input as bb_encode_int8_transposed_typed (vector path: in 16-byte
 * aligned for BB_F32 / BB_F64, 8-byte for BB_F16 / BB_BF16). */
int bb_encode_int8_timefirst_typed(const void *in, int32_t in_dtype,
                                   void *dst, const int64_t *unit_offset,
                                   int64_t nunit, int64_t nsample,
                                   int32_t nchan, int32_t npol,
                                   int32_t item_nbytes, void *stream);

/* ------------------------------------------------------- header batches
 * VDIF: extract the bit-fields of baseband/vdif/header.py:529-542, :557-559
 * (generic extractor baseband/base/header.py:35-87) for `nframe` headers at
 * src + frame_offset[i] (or i*frame_stride if frame_offset is NULL) into
 * fields[f * nframe + i], f indexing bb_vdif_field.  Then build the unit
 * table of a regular stream: frames_per_set consecutive frames form a set
 * (baseband/vdif/frame.py:201-243); slot = thread_slot[thread_id] (device
 * int32[1024], -1 = thread not selected, baseband/vdif/base.py:464-490);
 * unit_offset[set*nthread + slot] = payload offset, or -1 if invalid_data
 * (baseband/vdif/frame.py:79-90).  *n_inconsistent (device int32) counts
 * frames whose frame_nr differs from the first frame of their set or
 * whose slot is duplicated or missing, so the host can fall back to its
 * frame index (baseband/vdif/base.py:536-755).  The counter ACCUMULATES over
 * calls (the caller zeroes it), so one read needs one look at it.
 * Frame-index check (`VDIFStreamBase._get_index`,
 * baseband/vdif/base.py:386-390; the read-ahead verification of
 * baseband/base/base.py:1083-1125): with frames_per_second > 0 the first
 * frame of set s must satisfy
 *   (seconds - seconds0) * frames_per_second + frame_nr - frame_nr0
 *       == index0 + s
 * (seconds0 / frame_nr0 = fields of the stream's first header, index0 = frame
 * index of the first set handed in), else it is counted as inconsistent.
 * `fields` may be NULL when only the unit table is wanted. */
typedef enum bb_vdif_field {
    BB_VDIF_INVALID = 0, BB_VDIF_LEGACY, BB_VDIF_SECONDS, BB_VDIF_REF_EPOCH,
    BB_VDIF_FRAME_NR, BB_VDIF_VERSION, BB_VDIF_LG2_NCHAN,
    BB_VDIF_FRAME_LENGTH, BB_VDIF_COMPLEX, BB_VDIF_BITS_PER_SAMPLE,
    BB_VDIF_THREAD_ID, BB_VDIF_STATION_ID, BB_VDIF_EDV, BB_VDIF_WORD4,
    BB_VDIF_WORD5, BB_VDIF_WORD6, BB_VDIF_WORD7, BB_VDIF_NFIELD
} bb_vdif_field;
int bb_vdif_scan(const void *src, const int64_t *frame_offset,
                 int64_t frame_stride, int64_t nframe, int32_t header_nbytes,
                 int32_t frames_per_set, int32_t nthread,
                 const int32_t *thread_slot, int32_t *fields,
                 int64_t *unit_offset, int32_t *n_inconsistent,
                 int64_t index0, int32_t seconds0, int32_t frame_nr0,
                 int32_t frames_per_second, void *stream);

/* Mark 5B: header fields (baseband/mark5b/header.py:60-68), BCD decode
 * (baseband/base/utils.py:18-34, header.py:192-233 incl. the 156250 ns
 * "unrounding") and payload validity = not all 2500 words equal 0x11223344
 * (baseband/mark5b/frame.py:62-72).  unit_offset[i] = payload offset or -1.
 * Frame-index check (`Mark5BStreamBase._get_index`,
 * baseband/mark5b/base.py:206-213): with frames_per_second > 0 and
 * n_inconsistent non-NULL, frame i is counted in *n_inconsistent (accumulating
 * device int32) unless its sync word is 0xABADDEED, its BCD time is valid and
 *   (seconds - seconds0 + 86400 * dday) * frames_per_second
 *       + frame_nr - frame_nr0 == index0 + i,
 * dday = jday - jday0 wrapped into [-500, 500).  `fields` may be NULL.
 * A negative frame_offset[i] marks a frame the stream's index knows to be
 * absent: unit_offset[i] = -1, fields 0, nothing is read. */
typedef enum bb_mark5b_field {
    BB_M5B_SYNC = 0, BB_M5B_USER, BB_M5B_INTERNAL_TVG, BB_M5B_FRAME_NR,
    BB_M5B_BCD_JDAY, BB_M5B_BCD_SECONDS, BB_M5B_BCD_FRACTION, BB_M5B_CRC,
    BB_M5B_JDAY, BB_M5B_SECONDS, BB_M5B_FRACTION_NS, BB_M5B_VALID,
    BB_M5B_NFIELD
} bb_mark5b_field;
int bb_mark5b_scan(const void *src, const int64_t *frame_offset,
                   int64_t frame_stride, int64_t nframe, int32_t *fields,
                   int64_t *unit_offset, int32_t *n_inconsistent,
                   int64_t index0, int32_t jday0, int32_t seconds0,
                   int32_t frame_nr0, int32_t frames_per_second,
                   void *stream);

/* Mark 4: track-header bit transpose (`stream2words`,
 * baseband/mark4/header.py:47-63) for one chosen track -> 5 words per frame
 * in words5[i*5 + w], and frame validity = no error flag on any track
 * (baseband/mark4/frame.py:78-87).  unit_offset[i] = payload offset or -1.
 * Frame-index check (the time-based `_get_index` of
 * baseband/base/base.py:497-502 on the BCD time code,
 * baseband/mark4/header.py:223-262): with tick_step > 0 and n_inconsistent
 * non-NULL, frame i is counted in *n_inconsistent (accumulating) unless the
 * time code of `track` (unit year, day of year, h, m, s, ms) is that of
 * tick0 + tick_step * (index0 + i) quarter-milliseconds after 00:00 of MJD
 * mjd0.  `words5` may be NULL.  A negative frame_offset[i] marks an absent
 * frame (unit_offset[i] = -1, nothing read). */
int bb_mark4_scan(const void *src, const int64_t *frame_offset,
                  int64_t frame_stride, int64_t nframe, int32_t ntrack,
                  int32_t track, uint32_t *words5, int64_t *unit_offset,
                  int32_t *n_inconsistent, int64_t index0, int32_t mjd0,
                  int64_t tick0, int64_t tick_step, void *stream);

/* Writer-side frame assembly (the per-frame loop of StreamWriterBase.write,
 * baseband/base/base.py:1190-1262, which writes header + payload frame by
 * frame): header i (`headers + i * header_nbytes`, device memory, built by
 * the host from header0 and the frame index) is copied to
 * `dst + i * frame_stride`, and
 *   unit_offset[i * units_per_frame + u]
 *       = i * frame_stride + header_nbytes + u * unit_stride
 * is written for the encode call that follows.  With `valid` (device uint8
 * per frame) non-NULL, the payload of a frame with valid[i] == 0 is filled
 * with `fill_word` and its units are set to -1 so that the encode skips it
 * (Mark 5B: fill pattern 0x11223344, baseband/mark5b/frame.py:126-133).
 * `unit_offset` may be NULL. */
int bb_frames_assemble(void *dst, int64_t nframe, int64_t frame_stride,
                       int32_t header_nbytes, const void *headers,
                       const uint8_t *valid, uint32_t fill_word,
                       int64_t payload_nbytes, int32_t units_per_frame,
                       int64_t unit_stride, int64_t *unit_offset,
                       void *stream);

/* ---------------------------------------------------------- host ingest
 * File -> pinned staging on a persistent pool of native threads (the
 * reference reads each payload with one fh.readinto,
 * baseband/base/payload.py:83-143).  bb_host_copy: memcpy in up to `nthreads`
 * slices (e.g. out of a read-only mmap of the file: the page cache itself);
 * bb_host_pread: the same with pread(2) from a file descriptor, *nread =
 * bytes read before the first short slice.  No CUDA involved. */
int bb_host_copy(void *dst, const void *src, int64_t nbytes, int32_t nthreads);
/* The same without blocking the caller: bb_host_copy_begin hands the slices
 * to the pool and returns; bb_host_copy_wait blocks until they are done
 * (*nbytes = bytes copied; may be NULL).  One copy in flight at a time, begun
 * and waited for by the same thread: the readers use it to fill the next
 * chunk's staging buffer while they queue the current chunk's GPU work. */
int bb_host_copy_begin(void *dst, const void *src, int64_t nbytes,
                       int32_t nthreads);
int bb_host_copy_wait(int64_t *nbytes);
int bb_host_pread(int32_t fd, void *dst, int64_t nbytes, int64_t offset,
                  int32_t nthreads, int64_t *nread);

/* ------------------------------------------ frame location and frame index
 * The device-side replacement for the reference's sync search and frame
 * bookkeeping of irregular streams (`locate_frames`,
 * baseband/base/base.py:181-335; `RawOffsets`, baseband/base/offsets.py:6-126;
 * the per-frame repair of baseband/vdif/base.py:536-755 and the read-ahead
 * verification of baseband/base/base.py:1083-1219).
 *
 * bb_locate_frames: every byte position loc in [0, own_stop) of the device
 * region src[0, nbytes) where the masked pattern (host arrays of
 * pattern_nbytes <= 256 bytes; mask NULL = all ones) occurs at
 * loc + pattern_offset AND -- with frame_nbytes > 0 and check != 0 -- again
 * at loc + pattern_offset + check * frame_nbytes if that position lies inside
 * the region (the reference's `check=1`).  With at_eof != 0 the region ends
 * the file: frames must fit in it and a check position beyond it is not
 * required; otherwise a position whose check cannot be seen is left to the
 * next (overlapping) region.  base + loc is appended (atomically, unordered)
 * to locations[0, max_locations); *count (device int32, caller-zeroed)
 * receives the number found, which may exceed max_locations.  Positions that
 * hold the pattern and fit but FAIL the check go to `unverified` (same
 * conventions; may be NULL): the caller may still accept the last frame
 * before trailing damage, as the reference does by ending a stream at its
 * last good header (baseband/vdif/base.py:493-519).
 *
 * Frame table: uint64 entries, bb_index_table_init sets them to "empty".
 * bb_vdif_index / bb_mark5b_index read the header at every location found
 * (src = device copy of the file bytes from offset `base` on), compute its
 * frame index relative to the stream's first header
 *   VDIF    (seconds - seconds0) * fps + frame_nr - frame_nr0, slot from
 *           thread_slot[thread_id]        (baseband/vdif/base.py:386-390)
 *   Mark 5B (seconds - seconds0 + 86400 * dday) * fps + frame_nr - frame_nr0,
 *           BCD jday / seconds, dday = jday - jday0 wrapped to [-500, 500)
 *                                        (baseband/mark5b/base.py:206-213)
 *   Mark 4  time code of one track (unit year, day of year, h, m, s, ms:
 *           baseband/mark4/header.py:223-262) in 0.25 ms ticks relative to the
 *           first header (year0, yday0, tick0 = its tick within its day),
 *           divided by tick_step; year digit within +-1 year of year0; with
 *           check_crc the track's CRC-12 must hold (the all-ones sync also
 *           matches next to the true frame start when neighbouring header
 *           bits are set; the CRC tells them apart)
 * and keep, per (index, slot), the frame that comes first in the file
 * (atomicMin of 2 * offset + invalid flag).  stats (device int32[4],
 * caller-zeroed): [3] (VDIF) largest index among the frames of thread
 * `thread0`, the first header's: where the reference ends the stream
 * (`_last_header`, baseband/vdif/base.py:493-519); [0] largest index seen, [1] frames outside
 * [0, nset_max), [2] headers with an invalid BCD time (Mark 4: or a time off
 * the frame grid).
 * bb_index_table_finish turns the table into int64 byte offsets of the
 * frames, -1 where a frame is missing or flagged invalid: the
 * `frame_offset` / unit tables the scan and decode kernels take. */
int bb_locate_frames(const void *src, int64_t nbytes, int64_t own_stop,
                     const uint8_t *pattern, const uint8_t *mask,
                     int32_t pattern_nbytes, int64_t pattern_offset,
                     int64_t frame_nbytes, int32_t check, int32_t at_eof,
                     int64_t base, int64_t *locations, int32_t max_locations,
                     int32_t *count, int64_t *unverified,
                     int32_t max_unverified, int32_t *count_unverified,
                     void *stream);
int bb_index_table_init(uint64_t *table, int64_t nentry, void *stream);
int bb_vdif_index(const void *src, int64_t base, const int64_t *locations,
                  const int32_t *count, int32_t max_locations,
                  const int32_t *thread_slot, int32_t nthread,
                  int32_t seconds0, int32_t frame_nr0,
                  int32_t frames_per_second, int32_t thread0,
                  int64_t nset_max, uint64_t *table, int32_t *stats,
                  void *stream);
int bb_mark5b_index(const void *src, int64_t base, const int64_t *locations,
                    const int32_t *count, int32_t max_locations,
                    int32_t jday0, int32_t seconds0, int32_t frame_nr0,
                    int32_t frames_per_second, int64_t nset_max,
                    uint64_t *table, int32_t *stats, void *stream);
int bb_mark4_index(const void *src, int64_t base, const int64_t *locations,
                   const int32_t *count, int32_t max_locations,
                   int32_t ntrack, int32_t track, int32_t year0,
                   int32_t yday0, int32_t days_year0, int32_t days_prev_year,
                   int64_t tick0, int64_t tick_step, int32_t check_crc,
                   int64_t nset_max, uint64_t *table, int32_t *stats,
                   void *stream);
int bb_index_table_finish(const uint64_t *table, int64_t nentry,
                          int64_t *offsets, void *stream);

/* ------------------------------------------------- consumers on the device
 * The plug-in point for analysis that follows the decode is
 * baseband/tasks/__init__.py:25-62 (entry-point group 'baseband.tasks', the
 * baseband-tasks package: Square, Integrate, ...).  A consumer that runs on
 * the GPU need not see float32 samples at all:
 *
 * bb_state_counts accumulates, straight from the packed payloads,
 *   counts[bin][thread][elem][code] += number of samples with that code
 * (uint64, device memory, nbin x nthread x nelem x 2**bps, caller-zeroed) for
 * the frame sets of this call.  Set s of the call belongs to integration bin
 * (set_origin + s) / sets_per_bin; units at offset < 0 (invalid frames) are
 * left out, so sum_c counts = valid samples.  `code` is the bit field the
 * decoders look up in the level table (sample i of a word in bits
 * [i*bps, (i+1)*bps), element fastest: baseband/vdif/payload.py:53-63), hence
 *   sum over a bin of decoded**2 == sum_c counts[..., c] * levels[c]**2,
 * i.e. integrated power (Integrate(Square(fh))) and the digitiser statistics
 * follow from one pass over the packed bytes.  bps 1, 2, 4; nelem a power of
 * two; exact integer arithmetic (bit-identical for any launch shape). */
int bb_state_counts(const void *src, const int64_t *unit_offset, int64_t nset,
                    int32_t nthread, int64_t payload_nbytes, int32_t bps,
                    int32_t nelem, int64_t set_origin, int64_t sets_per_bin,
                    uint64_t *counts, int64_t nbin, void *stream);

/* The same for 8-bit two's-complement payloads (GUPPI, DADA;
 * baseband/guppi/payload.py:25-48): instead of a histogram,
 *   moments[bin][thread][elem][0..2] += (number of samples, sum, sum of
 *   squares)
 * as int64 (caller-zeroed): power (sum of squares / n), mean and variance per
 * integration bin, exact.  elem = byte index within a sample (nelem a power of
 * two, <= 1024); for channels-first GUPPI a unit is one channel row of a
 * frame, so `thread` is the channel and elem = (pol, re/im). */
int bb_int8_moments(const void *src, const int64_t *unit_offset, int64_t nset,
                    int32_t nthread, int64_t payload_nbytes, int32_t nelem,
                    int64_t set_origin, int64_t sets_per_bin,
                    int64_t *moments, int64_t nbin, void *stream);

/* bb_mark4_state_counts: the same for Mark 4 track words.  Frames are the
 * units: unit_offset[i] is the offset of frame i's payload (past the 160
 * header steps, as bb_mark4_scan writes it; < 0: invalid frame, left out);
 * frame i belongs to bin (set_origin + i) / sets_per_bin.
 *   counts[bin][chan][2 * sign + magnitude]   (nbin x nchan x 4, caller-zeroed)
 * indexed like the level table of bb_mark4_decode (baseband/mark4/payload.py:
 * 88-115), so integrated power = sum_c counts[..., c] * levels[c]**2.  The
 * five track layouts of bb_mark4_decode (nchan, fanout, ft). */
int bb_mark4_state_counts(const void *src, const int64_t *unit_offset,
                          int64_t nframe, int32_t nchan, int32_t fanout,
                          int32_t ft, int64_t set_origin, int64_t sets_per_bin,
                          uint64_t *counts, int64_t nbin, void *stream);

/* ------------------------------------------------------ bandwidth probes
 * Not part of the reference's path: the ceilings bench.py quotes next to the
 * decode kernels, measured in the same run with the kernels' own launch shape
 * (one-shot grid, 8 float4 per thread).  bb_probe_fill writes nbytes of
 * float32 1.0 (pattern 0: every warp store 512 contiguous bytes; pattern 1:
 * 8 pieces of 64 bytes per warp store, the row-group shape); bb_probe_copy is
 * a 16-byte-vector copy (read + write). */
int bb_probe_fill(void *dst, int64_t nbytes, int32_t pattern, void *stream);
int bb_probe_copy(void *dst, const void *src, int64_t nbytes, void *stream);
/* bb_probe_expand: the ceiling for a 1:16 expanding stream (2 bit -> float32)
 * with ideal access patterns: reads nbytes / 16 bytes of src and writes nbytes
 * of dst (pattern 0: contiguous input; 1: input in 16 interleaved streams, the
 * shape of a 16-thread VDIF frame set; 2: contiguous input wrapped to one MiB,
 * i.e. always an L2 hit; 3: a 1:4 stream instead, 8 bit -> float32, reading
 * nbytes / 4 bytes of contiguous input; 4: pattern 0 with leader threads
 * prefetching the next wave's input into L2 in bursts, BB_PROBE_LEAD /
 * BB_PROBE_AHEAD CTAs).  nbytes a multiple of 4096. */
int bb_probe_expand(void *dst, int64_t nbytes, const void *src,
                    int32_t pattern, void *stream);
/* bb_probe_prefetch: a pure-read phase that pulls nbytes of src into L2
 * (prefetch.global.L2::evict_last), for phased read-then-write experiments. */
int bb_probe_prefetch(const void *src, int64_t nbytes, void *stream);
/* bb_probe_read: read nbytes of src with the same launch shape and store
 * nothing: the pure-read rate, the ceiling of the consumers that only read
 * packed bytes (bb_state_counts, bb_int8_moments). */
int bb_probe_read(const void *src, int64_t nbytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BASEBAND_B200_H */
