"""Thin Python wrappers over the C ABI, using torch for device memory/streams.

Every function takes CUDA ``torch.Tensor`` buffers, passes raw pointers and
the current torch stream to ``libbaseband_b200.so`` and returns a tensor.
torch is plumbing only: all arithmetic happens in the hand-written kernels.
There is no CPU path; CPU tensors are rejected.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import (CODEC_LEVELS, CODEC_SINT, QUANT_OFFSET_BINARY,  # noqa
                   QUANT_MARK5B, QUANT_SINT, F32, F64, F16, BF16)

_FLOATP = ctypes.POINTER(ctypes.c_float)

# Counter of kernel-launching C calls, for bench.py's ``gpu_launches`` claim.
launch_count = 0


def _count(n=1):
    global launch_count
    launch_count += n


class _Here:
    """No-op guard: the device is already current."""
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_HERE = _Here()


def _on(device):
    """Device guard for a C call; free when ``device`` is already current
    (the per-call cost of ``torch.cuda.device`` showed in small reads)."""
    index = device.index
    if index is None or torch._C._cuda_getDevice() == index:
        return _HERE
    return torch.cuda.device(device)


def _stream_ptr(device):
    index = device.index
    if index is None:
        index = torch._C._cuda_getDevice()
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(index))


def _dev(t, name, dtype=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError('{} must be a CUDA torch.Tensor (there is no CPU '
                        'fallback)'.format(name))
    if dtype is not None and t.dtype != dtype:
        raise TypeError('{} must have dtype {}'.format(name, dtype))
    if not t.is_contiguous():
        raise ValueError('{} must be contiguous'.format(name))
    return ctypes.c_void_p(t.data_ptr())


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and (not isinstance(t, torch.Tensor)
                              or not t.is_cuda):
            raise TypeError('arguments must be CUDA torch.Tensors (there is '
                            'no CPU fallback)')


def _float_code(data):
    """bb_dtype of a float32/float64 tensor; anything else is refused (the
    kernels read 4 or 8 bytes per element)."""
    if data.dtype == torch.float32:
        return F32
    if data.dtype == torch.float64:
        return F64
    raise TypeError('data must be float32 or float64, not {}'.format(
        data.dtype))


# Element types the decoders can write (bb_dtype codes).
OUT_DTYPES = {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16}


def _typed(lib, name, out):
    """The decode entry point for ``out``'s element type and the arguments
    that select it: ``(fn, extra)``, where float32 uses the plain function
    (no extra argument) and float16 / bfloat16 its ``_typed`` variant, which
    takes the bb_dtype code before ``out``."""
    if out.dtype == torch.float32:
        return getattr(lib, name), ()
    code = OUT_DTYPES.get(out.dtype)
    if code is None:
        raise TypeError('out must be float32, float16 or bfloat16, not {}'
                        .format(out.dtype))
    try:
        fn = getattr(lib, name + '_typed')
    except AttributeError:
        raise ImportError('libbaseband_b200.so has no {}_typed: rebuild it '
                          'for float16 / bfloat16 output'.format(name))
    return fn, (code,)


# Element types the encoders can read (bb_dtype codes).
IN_DTYPES = {torch.float32: F32, torch.float64: F64, torch.float16: F16,
             torch.bfloat16: BF16}


def _typed_encoder(lib, name, data):
    """The encode entry point for ``data``'s element type and its bb_dtype
    code: ``(fn, code)``.  float32 / float64 use the plain function, float16
    / bfloat16 its ``_typed`` variant, which takes the same arguments."""
    code = IN_DTYPES.get(data.dtype)
    if code is None:
        raise TypeError('data must be float32, float64, float16 or bfloat16, '
                        'not {}'.format(data.dtype))
    if code in (F32, F64):
        return getattr(lib, name), code
    try:
        return getattr(lib, name + '_typed'), code
    except AttributeError:
        raise ImportError('libbaseband_b200.so has no {}_typed: rebuild it '
                          'for float16 / bfloat16 input'.format(name))


def _levels_arg(levels):
    if levels is None:
        return None, None
    lv = np.ascontiguousarray(levels, dtype=np.float32)
    return lv, lv.ctypes.data_as(_FLOATP)


def to_device_bytes(raw, device, pinned=None):
    """numpy/bytes -> uint8 CUDA tensor (async copy on the current stream
    when the source is pinned)."""
    if isinstance(raw, torch.Tensor):
        return raw.to(device, non_blocking=True)
    arr = np.frombuffer(raw, np.uint8) if isinstance(
        raw, (bytes, bytearray, memoryview)) else np.ascontiguousarray(
            raw).view(np.uint8).reshape(-1)
    t = torch.from_numpy(arr) if arr.flags.writeable else torch.from_numpy(
        arr.copy())
    return t.to(device, non_blocking=True)


def decode_bitfield(src, unit_offset, nset, nthread, payload_nbytes, bps,
                    nelem, complex_data=False, codec=CODEC_LEVELS,
                    levels=None, fill_value=0.0, sample_start=0,
                    nsample=None, out=None, dtype=torch.float32):
    """bb_decode_bitfield -> tensor (nsample, nthread, nelem) of ``dtype``
    (float32, float16 or bfloat16) or of ``out``'s dtype."""
    lib = _lib.load()
    _require_cuda(src, unit_offset, out)
    spf = payload_nbytes * 8 // (bps * nelem)
    if nsample is None:
        nsample = nset * spf - sample_start
    if out is None:
        out = torch.empty((nsample, nthread, nelem), dtype=dtype,
                          device=src.device)
    elif out.numel() != nsample * nthread * nelem:
        raise ValueError('out has the wrong number of elements')
    if out.numel() == 0:
        return out                       # an empty tensor has no storage
    fn, typed = _typed(lib, 'bb_decode_bitfield', out)
    keep, lv = _levels_arg(levels)
    with _on(src.device):
        rc = fn(
            _dev(src, 'src', torch.uint8), _dev(unit_offset, 'unit_offset',
                                                torch.int64),
            nset, nthread, payload_nbytes, bps, nelem, int(bool(complex_data)),
            codec, lv, float(fill_value), sample_start, nsample, *typed,
            _dev(out, 'out'), _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()
    return out


def _select_entry(lib, name, out):
    """A selective decode entry point and the bb_dtype code of ``out``."""
    code = OUT_DTYPES.get(out.dtype)
    if code is None:
        raise TypeError('out must be float32, float16 or bfloat16, not {}'
                        .format(out.dtype))
    try:
        return getattr(lib, name), code
    except AttributeError:
        raise ImportError('libbaseband_b200.so has no {}: rebuild it for '
                          'subset reads'.format(name))


def decode_select_bitfield(src, unit_offset, nset, nthread, payload_nbytes,
                           bps, nelem, complex_data, codec, levels, fill_value,
                           sample_start, nsample, sel, out):
    """bb_decode_select_bitfield: only the components ``sel`` (int32 CUDA
    tensor of indices into the decoded row of `decode_bitfield`) of every
    row, ``out`` (float32, float16 or bfloat16) = (nsample, len(sel))."""
    lib = _lib.load()
    _require_cuda(src, unit_offset, sel, out)
    nsel = sel.numel()
    if out.numel() != nsample * nsel:
        raise ValueError('out has the wrong number of elements')
    if out.numel() == 0:
        return out
    fn, code = _select_entry(lib, 'bb_decode_select_bitfield', out)
    keep, lv = _levels_arg(levels)
    with _on(src.device):
        rc = fn(
            _dev(src, 'src', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nset, nthread,
            payload_nbytes, bps, nelem, int(bool(complex_data)), codec, lv,
            float(fill_value), sample_start, nsample,
            _dev(sel, 'sel', torch.int32), nsel, code, _dev(out, 'out'),
            _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()
    return out


def decode_select_int8(src, unit_offset, nunit, nsample, heap, heap_stride,
                       t_stride, off, t_begin, t_end, out_t0, out):
    """bb_decode_select_int8: component j of sample t of unit u is the int8
    at ``unit_offset[u] + (t // heap) * heap_stride + (t % heap) * t_stride
    + off[j]`` (``off``: int32 CUDA tensor); samples [t_begin[u], t_end[u])
    go to rows out_t0[u] on of ``out`` (float32, float16 or bfloat16, rows
    of len(off))."""
    lib = _lib.load()
    _require_cuda(src, unit_offset, off, t_begin, t_end, out_t0, out)
    if out.numel() == 0:
        return out
    fn, code = _select_entry(lib, 'bb_decode_select_int8', out)
    with _on(src.device):
        rc = fn(
            _dev(src, 'src', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nunit, nsample,
            heap, heap_stride, t_stride, _dev(off, 'off', torch.int32),
            off.numel(), _dev(t_begin, 't_begin', torch.int64),
            _dev(t_end, 't_end', torch.int64),
            _dev(out_t0, 'out_t0', torch.int64), code, _dev(out, 'out'),
            _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()
    return out


def encode_bitfield(data, dst, unit_offset, nset, nthread, payload_nbytes,
                    bps, nelem, quantiser=QUANT_OFFSET_BINARY):
    """bb_encode_bitfield: quantise+pack ``data`` (float32, float64, float16
    or bfloat16, logical shape (nset*spf, nthread, nelem)) into ``dst``
    (uint8) at the unit offsets.  A 16-bit value encodes as its float32
    value does."""
    lib = _lib.load()
    _require_cuda(data, dst, unit_offset)
    fn, code = _typed_encoder(lib, 'bb_encode_bitfield', data)
    if data.numel() == 0:
        return dst                      # nothing to encode
    with _on(dst.device):
        rc = fn(
            _dev(data, 'data'), code, _dev(dst, 'dst', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nset, nthread,
            payload_nbytes, bps, nelem, quantiser, _stream_ptr(dst.device))
    _lib.check(rc, lib)
    _count()
    return dst


def mark4_decode(src, unit_offset, nframe, nchan, fanout, ft=False,
                 levels=None, fill_value=0.0, sample_start=0, nsample=None,
                 out=None, dtype=torch.float32):
    """bb_mark4_decode -> tensor (nsample, nchan) of ``dtype`` (float32,
    float16 or bfloat16) or of ``out``'s dtype."""
    lib = _lib.load()
    spf = 20000 * fanout
    if nsample is None:
        nsample = nframe * spf - sample_start
    if out is None:
        out = torch.empty((nsample, nchan), dtype=dtype, device=src.device)
    if out.numel() == 0:
        return out
    fn, typed = _typed(lib, 'bb_mark4_decode', out)
    keep, lv = _levels_arg(levels)
    with _on(src.device):
        rc = fn(
            _dev(src, 'src', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nframe, nchan,
            fanout, int(bool(ft)), lv, float(fill_value), sample_start,
            nsample, *typed, _dev(out, 'out'), _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()
    return out


def mark4_encode(data, dst, unit_offset, nframe, nchan, fanout, ft=False):
    """bb_mark4_encode of ``data`` (float32, float64, float16 or
    bfloat16)."""
    lib = _lib.load()
    fn, code = _typed_encoder(lib, 'bb_mark4_encode', data)
    if data.numel() == 0:
        return dst                      # nothing to encode
    with _on(dst.device):
        rc = fn(
            _dev(data, 'data'), code, _dev(dst, 'dst', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nframe, nchan,
            fanout, int(bool(ft)), _stream_ptr(dst.device))
    _lib.check(rc, lib)
    _count()
    return dst


def mark4_decode_words(words, nword, nchan, fanout, ft=False, levels=None,
                       out=None):
    lib = _lib.load()
    if out is None:
        out = torch.empty((nword * fanout, nchan), dtype=torch.float32,
                          device=words.device)
    keep, lv = _levels_arg(levels)
    with _on(words.device):
        rc = lib.bb_mark4_decode_words(
            _dev(words, 'words'), nword, nchan, fanout, int(bool(ft)), lv,
            _dev(out, 'out', torch.float32), _stream_ptr(words.device))
    _lib.check(rc, lib)
    _count()
    return out


def mark4_encode_words(data, words, nword, nchan, fanout, ft=False):
    lib = _lib.load()
    code = _float_code(data)
    if data.numel() == 0:
        return words                      # nothing to encode
    with _on(words.device):
        rc = lib.bb_mark4_encode_words(
            _dev(data, 'data'), code, _dev(words, 'words'), nword, nchan,
            fanout, int(bool(ft)), _stream_ptr(words.device))
    _lib.check(rc, lib)
    _count()
    return words


def decode_int8_transposed(src, unit_offset, nunit, nrow, ncol, item_nbytes,
                           col_begin, col_end, out_col0, out):
    """bb_decode_int8_transposed into ``out`` (float32, float16 or
    bfloat16)."""
    lib = _lib.load()
    if out.numel() == 0:
        return out
    fn, typed = _typed(lib, 'bb_decode_int8_transposed', out)
    with _on(src.device):
        rc = fn(
            _dev(src, 'src', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nunit, nrow, ncol,
            item_nbytes, _dev(col_begin, 'col_begin', torch.int64),
            _dev(col_end, 'col_end', torch.int64),
            _dev(out_col0, 'out_col0', torch.int64), *typed,
            _dev(out, 'out'), _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()
    return out


def encode_int8_transposed(data, dst, unit_offset, nunit, nrow, ncol,
                           item_nbytes):
    """bb_encode_int8_transposed of ``data`` (float32, float64, float16 or
    bfloat16)."""
    lib = _lib.load()
    fn, code = _typed_encoder(lib, 'bb_encode_int8_transposed', data)
    if data.numel() == 0:
        return dst                      # nothing to encode
    with _on(dst.device):
        rc = fn(
            _dev(data, 'data'), code, _dev(dst, 'dst', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nunit, nrow, ncol,
            item_nbytes, _stream_ptr(dst.device))
    _lib.check(rc, lib)
    _count()
    return dst


def decode_int8_timefirst(src, unit_offset, nunit, nsample, nchan, npol,
                          item_nbytes, t_begin, t_end, out_t0, out):
    """bb_decode_int8_timefirst: [time][chan][pol] int8 -> (time, pol, chan)
    rows of ``out`` (float32, float16 or bfloat16)."""
    lib = _lib.load()
    if out.numel() == 0:
        return out
    fn, typed = _typed(lib, 'bb_decode_int8_timefirst', out)
    with _on(src.device):
        rc = fn(
            _dev(src, 'src', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nunit, nsample,
            nchan, npol, item_nbytes, _dev(t_begin, 't_begin', torch.int64),
            _dev(t_end, 't_end', torch.int64),
            _dev(out_t0, 'out_t0', torch.int64), *typed,
            _dev(out, 'out'), _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()
    return out


def encode_int8_timefirst(data, dst, unit_offset, nunit, nsample, nchan, npol,
                          item_nbytes):
    """bb_encode_int8_timefirst of ``data`` (float32, float64, float16 or
    bfloat16)."""
    lib = _lib.load()
    fn, code = _typed_encoder(lib, 'bb_encode_int8_timefirst', data)
    if data.numel() == 0:
        return dst                      # nothing to encode
    with _on(dst.device):
        rc = fn(
            _dev(data, 'data'), code, _dev(dst, 'dst', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nunit, nsample,
            nchan, npol, item_nbytes, _stream_ptr(dst.device))
    _lib.check(rc, lib)
    _count()
    return dst


VDIF_NFIELD = 17
# row indices of the ``fields`` array (enum bb_vdif_field / bb_mark5b_field)
(VDIF_INVALID, VDIF_LEGACY, VDIF_SECONDS, VDIF_REF_EPOCH, VDIF_FRAME_NR,
 VDIF_VERSION, VDIF_LG2_NCHAN, VDIF_FRAME_LENGTH, VDIF_COMPLEX,
 VDIF_BITS_PER_SAMPLE, VDIF_THREAD_ID, VDIF_STATION_ID, VDIF_EDV, VDIF_WORD4,
 VDIF_WORD5, VDIF_WORD6, VDIF_WORD7) = range(17)
(M5B_SYNC, M5B_USER, M5B_INTERNAL_TVG, M5B_FRAME_NR, M5B_BCD_JDAY,
 M5B_BCD_SECONDS, M5B_BCD_FRACTION, M5B_CRC, M5B_JDAY, M5B_SECONDS,
 M5B_FRACTION_NS, M5B_VALID) = range(12)
M5B_NFIELD = 12


def zeros(shape, dtype, device):
    """Zeroed device tensor by ``bb_memset`` (a memset on the current stream,
    not a fill kernel)."""
    lib = _lib.load()
    t = torch.empty(shape, dtype=dtype, device=device)
    if t.numel():
        with _on(t.device):
            _lib.check(lib.bb_memset(ctypes.c_void_p(t.data_ptr()), 0,
                                     t.numel() * t.element_size(),
                                     _stream_ptr(t.device)), lib)
    return t


def new_counter(device):
    """Zeroed device int32[1]: the accumulating inconsistency counter the scan
    kernels add to (one per reader, looked at once per ``read``)."""
    return zeros(1, torch.int32, device)


def vdif_scan(src, nframe, frame_stride, header_nbytes, frames_per_set,
              thread_slot, nthread, frame_offset=None, check=None, bad=None,
              want_fields=True):
    """bb_vdif_scan -> (fields int32 (NFIELD, nframe) or None, unit_offset
    int64 (nset*nthread,), n_inconsistent int32[1]).

    ``check = (index0, seconds0, frame_nr0, frames_per_second)`` folds the
    frame-index check into the scan; ``bad`` is an accumulating counter from
    `new_counter` (a fresh one is made if omitted)."""
    lib = _lib.load()
    dev = src.device
    fields = (torch.empty((VDIF_NFIELD, nframe), dtype=torch.int32,
                          device=dev) if want_fields else None)
    nset = nframe // frames_per_set
    unit_offset = torch.empty((max(nset * nthread, 1),), dtype=torch.int64,
                              device=dev)
    if nframe <= 0:
        unit_offset.fill_(-1)
    if bad is None:
        bad = new_counter(dev)
    index0, seconds0, frame_nr0, fps = check if check is not None \
        else (0, 0, 0, 0)
    with _on(dev):
        rc = lib.bb_vdif_scan(
            _dev(src, 'src', torch.uint8),
            None if frame_offset is None else _dev(frame_offset,
                                                   'frame_offset',
                                                   torch.int64),
            frame_stride, nframe, header_nbytes, frames_per_set, nthread,
            _dev(thread_slot, 'thread_slot', torch.int32),
            None if fields is None else _dev(fields, 'fields'),
            _dev(unit_offset, 'unit_offset'), _dev(bad, 'bad'),
            int(index0), int(seconds0), int(frame_nr0), int(fps),
            _stream_ptr(dev))
    _lib.check(rc, lib)
    _count(3)          # fill, scan, count-missing kernels
    return fields, unit_offset[:nset * nthread], bad


def mark5b_scan(src, nframe, frame_stride=10016, frame_offset=None,
                check=None, bad=None, want_fields=True):
    """bb_mark5b_scan -> (fields or None, unit_offset).  ``check = (index0,
    jday0, seconds0, frame_nr0, frames_per_second)`` with an accumulating
    counter ``bad`` folds the frame-index check into the scan."""
    lib = _lib.load()
    dev = src.device
    fields = (torch.empty((M5B_NFIELD, nframe), dtype=torch.int32,
                          device=dev) if want_fields else None)
    unit_offset = torch.empty((nframe,), dtype=torch.int64, device=dev)
    if check is not None and bad is None:
        raise ValueError('a frame-index check needs a counter')
    index0, jday0, seconds0, frame_nr0, fps = check if check is not None \
        else (0, 0, 0, 0, 0)
    with _on(dev):
        rc = lib.bb_mark5b_scan(
            _dev(src, 'src', torch.uint8),
            None if frame_offset is None else _dev(frame_offset,
                                                   'frame_offset',
                                                   torch.int64),
            frame_stride, nframe,
            None if fields is None else _dev(fields, 'fields'),
            _dev(unit_offset, 'unit_offset'),
            None if bad is None else _dev(bad, 'bad'), int(index0),
            int(jday0), int(seconds0), int(frame_nr0), int(fps),
            _stream_ptr(dev))
    _lib.check(rc, lib)
    _count()
    return fields, unit_offset


def mark4_scan(src, nframe, ntrack, frame_stride=None, track=0,
               frame_offset=None, check=None, bad=None, want_words=True):
    """bb_mark4_scan -> (words5 or None, unit_offset).  ``check = (index0,
    mjd0, tick0, tick_step)`` (quarter-millisecond ticks) with an
    accumulating counter ``bad`` folds the time-code check into the scan."""
    lib = _lib.load()
    dev = src.device
    if frame_stride is None:
        frame_stride = ntrack * 2500
    words5 = (torch.empty((nframe, 5), dtype=torch.int32, device=dev)
              if want_words else None)
    unit_offset = torch.empty((nframe,), dtype=torch.int64, device=dev)
    if check is not None and bad is None:
        raise ValueError('a time-code check needs a counter')
    index0, mjd0, tick0, tick_step = check if check is not None \
        else (0, 0, 0, 0)
    with _on(dev):
        rc = lib.bb_mark4_scan(
            _dev(src, 'src', torch.uint8),
            None if frame_offset is None else _dev(frame_offset,
                                                   'frame_offset',
                                                   torch.int64),
            frame_stride, nframe, ntrack, track,
            None if words5 is None else _dev(words5, 'words5'),
            _dev(unit_offset, 'unit_offset'),
            None if bad is None else _dev(bad, 'bad'), int(index0),
            int(mjd0), int(tick0), int(tick_step), _stream_ptr(dev))
    _lib.check(rc, lib)
    _count()
    return words5, unit_offset


def frames_assemble(headers, frame_nbytes, payload_nbytes=0, valid=None,
                    fill_word=0, units_per_frame=1, unit_stride=0):
    """bb_frames_assemble -> (frames uint8 (nframe, frame_nbytes),
    unit_offset int64 (nframe * units_per_frame,)).

    ``headers``: uint8 CUDA tensor (nframe, header_nbytes), one header per
    frame; ``valid``: optional uint8 CUDA tensor (nframe,), frames with 0 get
    their payload filled with ``fill_word`` and unit offsets -1."""
    lib = _lib.load()
    dev = headers.device
    nframe, header_nbytes = headers.shape
    frames = torch.empty((nframe, frame_nbytes), dtype=torch.uint8,
                         device=dev)
    unit_offset = torch.empty((nframe * units_per_frame,), dtype=torch.int64,
                              device=dev)
    with _on(dev):
        rc = lib.bb_frames_assemble(
            _dev(frames, 'frames'), nframe, frame_nbytes, header_nbytes,
            _dev(headers, 'headers', torch.uint8),
            None if valid is None else _dev(valid, 'valid', torch.uint8),
            int(fill_word), int(payload_nbytes), int(units_per_frame),
            int(unit_stride), _dev(unit_offset, 'unit_offset'),
            _stream_ptr(dev))
    _lib.check(rc, lib)
    _count()
    return frames, unit_offset


def _host_bytes(values):
    """Byte view of a pattern: bytes stay bytes, integers are unsigned 32-bit
    little-endian words (`byte_array`, baseband/base/utils.py:251-270)."""
    arr = np.asarray(values)
    if arr.dtype.kind in 'iu' and arr.dtype.itemsize != 1:
        arr = arr.astype('<u4')
    arr = np.ascontiguousarray(arr).view(np.uint8).reshape(-1)
    return arr, arr.ctypes.data_as(ctypes.c_void_p)


def locate_frames(src, pattern, mask=None, frame_nbytes=0, pattern_offset=0,
                  own_stop=None, check=1, at_eof=True, base=0,
                  max_locations=None, unverified=None):
    """bb_locate_frames -> (locations int64 (max_locations,), count int32[1]),
    both on the device; ``locations[:count]`` are the (unordered) byte
    positions ``base + loc`` at which the masked pattern starts a frame.
    ``unverified = (locations, count)`` (device tensors, count accumulating)
    collects the positions that hold the pattern but fail the check."""
    lib = _lib.load()
    dev = src.device
    nbytes = src.numel()
    if own_stop is None:
        own_stop = nbytes
    pat, pat_p = _host_bytes(pattern)
    if mask is not None:
        msk, msk_p = _host_bytes(mask)
        if msk.size != pat.size:
            raise ValueError('mask and pattern must have the same size')
    else:
        msk_p = None
    if max_locations is None:
        # a sync pattern can match a few bytes either side of a frame start
        # as well: room for several candidates per frame
        max_locations = (8 * (nbytes // frame_nbytes + 2) if frame_nbytes
                         else 4096)
    locations = torch.empty((max(int(max_locations), 1),), dtype=torch.int64,
                            device=dev)
    count = zeros(1, torch.int32, dev)
    with _on(dev):
        rc = lib.bb_locate_frames(
            _dev(src, 'src', torch.uint8), nbytes, int(own_stop), pat_p,
            msk_p, pat.size, int(pattern_offset), int(frame_nbytes),
            int(check), int(bool(at_eof)), int(base),
            _dev(locations, 'locations'), int(max_locations),
            _dev(count, 'count'),
            None if unverified is None else _dev(unverified[0], 'unverified',
                                                 torch.int64),
            0 if unverified is None else unverified[0].numel(),
            None if unverified is None else _dev(unverified[1], 'count',
                                                 torch.int32),
            _stream_ptr(dev))
    _lib.check(rc, lib)
    _count()
    return locations, count


def index_table(nentry, device):
    """Empty frame table (bb_index_table_init): int64 storage of the uint64
    entries."""
    lib = _lib.load()
    table = torch.empty((int(nentry),), dtype=torch.int64, device=device)
    with _on(table.device):
        rc = lib.bb_index_table_init(_dev(table, 'table'), int(nentry),
                                     _stream_ptr(table.device))
    _lib.check(rc, lib)
    _count()
    return table


def vdif_index(src, base, locations, count, thread_slot, nthread, seconds0,
               frame_nr0, fps, nset_max, table, stats, thread0=-1):
    lib = _lib.load()
    with _on(src.device):
        rc = lib.bb_vdif_index(
            _dev(src, 'src', torch.uint8), int(base),
            _dev(locations, 'locations', torch.int64),
            _dev(count, 'count', torch.int32), locations.numel(),
            _dev(thread_slot, 'thread_slot', torch.int32), nthread,
            int(seconds0), int(frame_nr0), int(fps), int(thread0),
            int(nset_max), _dev(table, 'table', torch.int64),
            _dev(stats, 'stats', torch.int32), _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()


def mark5b_index(src, base, locations, count, jday0, seconds0, frame_nr0,
                 fps, nset_max, table, stats):
    lib = _lib.load()
    with _on(src.device):
        rc = lib.bb_mark5b_index(
            _dev(src, 'src', torch.uint8), int(base),
            _dev(locations, 'locations', torch.int64),
            _dev(count, 'count', torch.int32), locations.numel(), int(jday0),
            int(seconds0), int(frame_nr0), int(fps), int(nset_max),
            _dev(table, 'table', torch.int64),
            _dev(stats, 'stats', torch.int32), _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()


def mark4_index(src, base, locations, count, ntrack, track, year0, yday0,
                days_year0, days_prev_year, tick0, tick_step, nset_max, table,
                stats, check_crc=True):
    lib = _lib.load()
    with _on(src.device):
        rc = lib.bb_mark4_index(
            _dev(src, 'src', torch.uint8), int(base),
            _dev(locations, 'locations', torch.int64),
            _dev(count, 'count', torch.int32), locations.numel(), int(ntrack),
            int(track), int(year0), int(yday0), int(days_year0),
            int(days_prev_year), int(tick0), int(tick_step),
            int(bool(check_crc)), int(nset_max),
            _dev(table, 'table', torch.int64),
            _dev(stats, 'stats', torch.int32), _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()


def index_table_finish(table):
    """bb_index_table_finish -> int64 byte offsets, -1 = missing/invalid."""
    lib = _lib.load()
    offsets = torch.empty_like(table)
    with _on(table.device):
        rc = lib.bb_index_table_finish(
            _dev(table, 'table', torch.int64), table.numel(),
            _dev(offsets, 'offsets'), _stream_ptr(table.device))
    _lib.check(rc, lib)
    _count()
    return offsets


def state_counts(src, unit_offset, nset, nthread, payload_nbytes, bps, nelem,
                 counts, set_origin=0, sets_per_bin=None):
    """bb_state_counts: add the state counts of ``nset`` frame sets to
    ``counts`` (int64 CUDA tensor (nbin, nthread, nelem, 2**bps))."""
    lib = _lib.load()
    _require_cuda(src, unit_offset, counts)
    nbin = counts.shape[0]
    if tuple(counts.shape[1:]) != (nthread, nelem, 1 << bps):
        raise ValueError('counts must have shape (nbin, nthread, nelem, '
                         '2**bps)')
    if sets_per_bin is None:
        sets_per_bin = max(1, set_origin + nset)
    with _on(src.device):
        rc = lib.bb_state_counts(
            _dev(src, 'src', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nset, nthread,
            payload_nbytes, bps, nelem, int(set_origin), int(sets_per_bin),
            _dev(counts, 'counts', torch.int64), nbin,
            _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()
    return counts


def byte_counts(src, unit_offset, nset, nthread, payload_nbytes, nelem,
                counts, set_origin=0, sets_per_bin=None):
    """bb_byte_counts: add the counts of every stored byte value of ``nset``
    sets of 8-bit units to ``counts`` (int64 CUDA tensor (nbin, nthread,
    nelem, 256))."""
    lib = _lib.load()
    _require_cuda(src, unit_offset, counts)
    nbin = counts.shape[0]
    if tuple(counts.shape[1:]) != (nthread, nelem, 256):
        raise ValueError('counts must have shape (nbin, nthread, nelem, 256)')
    if sets_per_bin is None:
        sets_per_bin = max(1, set_origin + nset)
    with _on(src.device):
        rc = lib.bb_byte_counts(
            _dev(src, 'src', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nset, nthread,
            payload_nbytes, nelem, int(set_origin), int(sets_per_bin),
            _dev(counts, 'counts', torch.int64), nbin,
            _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()
    return counts


def mark4_state_counts(src, unit_offset, nframe, nchan, fanout, ft, counts,
                       set_origin=0, sets_per_bin=None):
    """bb_mark4_state_counts: add the (sign, magnitude) state counts of
    ``nframe`` Mark 4 frames (``unit_offset``: payload offsets as written by
    `mark4_scan`) to ``counts`` (int64 CUDA tensor (nbin, nchan, 4), indexed
    2 * sign + magnitude like `levels.sign_magnitude`)."""
    lib = _lib.load()
    _require_cuda(src, unit_offset, counts)
    nbin = counts.shape[0]
    if tuple(counts.shape[1:]) != (nchan, 4):
        raise ValueError('counts must have shape (nbin, nchan, 4)')
    if sets_per_bin is None:
        sets_per_bin = max(1, set_origin + nframe)
    with _on(src.device):
        rc = lib.bb_mark4_state_counts(
            _dev(src, 'src', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nframe, nchan,
            fanout, int(bool(ft)), int(set_origin), int(sets_per_bin),
            _dev(counts, 'counts', torch.int64), nbin,
            _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()
    return counts


def int8_moments(src, unit_offset, nset, nthread, payload_nbytes, nelem,
                 moments, set_origin=0, sets_per_bin=None):
    """bb_int8_moments: add (n, sum, sum of squares) of ``nset`` sets of
    8-bit units to ``moments`` (int64 CUDA tensor (nbin, nthread, nelem, 3))."""
    lib = _lib.load()
    _require_cuda(src, unit_offset, moments)
    nbin = moments.shape[0]
    if tuple(moments.shape[1:]) != (nthread, nelem, 3):
        raise ValueError('moments must have shape (nbin, nthread, nelem, 3)')
    if sets_per_bin is None:
        sets_per_bin = max(1, set_origin + nset)
    with _on(src.device):
        rc = lib.bb_int8_moments(
            _dev(src, 'src', torch.uint8),
            _dev(unit_offset, 'unit_offset', torch.int64), nset, nthread,
            payload_nbytes, nelem, int(set_origin), int(sets_per_bin),
            _dev(moments, 'moments', torch.int64), nbin,
            _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()
    return moments


def probe_fill(dst, pattern=0):
    """bb_probe_fill: write the whole tensor ``dst`` with the decode kernels'
    launch shape (pure-write bandwidth probe)."""
    lib = _lib.load()
    nbytes = dst.numel() * dst.element_size()
    with _on(dst.device):
        rc = lib.bb_probe_fill(_dev(dst, 'dst'), nbytes, pattern,
                               _stream_ptr(dst.device))
    _lib.check(rc, lib)
    _count()
    return dst


def probe_copy(dst, src):
    """bb_probe_copy: vector copy of ``src`` into ``dst`` (read + write)."""
    lib = _lib.load()
    nbytes = src.numel() * src.element_size()
    if dst.numel() * dst.element_size() != nbytes:
        raise ValueError('dst and src must have the same size')
    with _on(dst.device):
        rc = lib.bb_probe_copy(_dev(dst, 'dst'), _dev(src, 'src'), nbytes,
                               _stream_ptr(dst.device))
    _lib.check(rc, lib)
    _count()
    return dst


def probe_read(src):
    """bb_probe_read: read all of ``src`` and store nothing (pure-read
    bandwidth probe: the ceiling of the packed-byte consumers)."""
    lib = _lib.load()
    nbytes = src.numel() * src.element_size()
    with _on(src.device):
        rc = lib.bb_probe_read(_dev(src, 'src'), nbytes,
                               _stream_ptr(src.device))
    _lib.check(rc, lib)
    _count()


def probe_expand(dst, src, pattern=0):
    """bb_probe_expand: write all of ``dst`` from 1/16 as many bytes of
    ``src`` (the ceiling for a 2 bit -> float32 stream)."""
    lib = _lib.load()
    nbytes = dst.numel() * dst.element_size() // 4096 * 4096
    ratio = 4 if pattern == 3 else 16
    if src.numel() * src.element_size() < nbytes // ratio:
        raise ValueError('src too small')
    with _on(dst.device):
        rc = lib.bb_probe_expand(_dev(dst, 'dst'), nbytes, _dev(src, 'src'),
                                 pattern, _stream_ptr(dst.device))
    _lib.check(rc, lib)
    _count()
    return nbytes + nbytes // ratio
