"""ctypes binding of ``libbaseband_b200.so`` (see include/baseband_b200.h).

There is no CPU fallback: if the CUDA library has not been built, or a call
fails, the error is raised.  Status codes are mapped to the exception types
the reference raises for the same condition (SURVEY.md section 8(b)).
"""
import ctypes
import os
from ctypes import (POINTER, c_char_p, c_float, c_int, c_int32, c_int64,
                    c_uint32, c_void_p)

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libbaseband_b200.so')

BB_OK, BB_ERR_ARGUMENT, BB_ERR_ALIGNMENT, BB_ERR_UNSUPPORTED, BB_ERR_CUDA = (
    0, -1, -2, -3, -4)
CODEC_LEVELS, CODEC_SINT = 0, 1
QUANT_OFFSET_BINARY, QUANT_MARK5B, QUANT_SINT = 0, 1, 2
F32, F64, F16, BF16 = 0, 1, 2, 3

_pf = POINTER(c_float)
_pi64 = c_void_p      # device int64*
_pv = c_void_p

SIGNATURES = {
    'bb_abi_version': (c_int, []),
    'bb_last_error': (c_char_p, []),
    'bb_device_count': (c_int, []),
    'bb_set_device': (c_int, [c_int]),
    'bb_device_sm_count': (c_int, [c_int]),
    'bb_malloc': (c_int, [POINTER(c_void_p), c_int64]),
    'bb_free': (c_int, [c_void_p]),
    'bb_host_alloc': (c_int, [POINTER(c_void_p), c_int64]),
    'bb_host_free': (c_int, [c_void_p]),
    'bb_host_register': (c_int, [c_void_p, c_int64]),
    'bb_host_unregister': (c_int, [c_void_p]),
    'bb_memcpy_h2d': (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    'bb_memcpy_d2h': (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    'bb_memset': (c_int, [c_void_p, c_int, c_int64, c_void_p]),
    'bb_stream_create': (c_int, [POINTER(c_void_p)]),
    'bb_stream_destroy': (c_int, [c_void_p]),
    'bb_stream_synchronize': (c_int, [c_void_p]),
    'bb_decode_bitfield': (c_int, [
        _pv, _pi64, c_int64, c_int32, c_int64, c_int32, c_int32, c_int32,
        c_int32, _pf, c_float, c_int64, c_int64, _pv, c_void_p]),
    'bb_decode_bitfield_typed': (c_int, [
        _pv, _pi64, c_int64, c_int32, c_int64, c_int32, c_int32, c_int32,
        c_int32, _pf, c_float, c_int64, c_int64, c_int32, _pv, c_void_p]),
    'bb_encode_bitfield': (c_int, [
        _pv, c_int32, _pv, _pi64, c_int64, c_int32, c_int64, c_int32,
        c_int32, c_int32, c_void_p]),
    'bb_encode_bitfield_typed': (c_int, [
        _pv, c_int32, _pv, _pi64, c_int64, c_int32, c_int64, c_int32,
        c_int32, c_int32, c_void_p]),
    'bb_mark4_decode': (c_int, [
        _pv, _pi64, c_int64, c_int32, c_int32, c_int32, _pf, c_float,
        c_int64, c_int64, _pv, c_void_p]),
    'bb_mark4_decode_typed': (c_int, [
        _pv, _pi64, c_int64, c_int32, c_int32, c_int32, _pf, c_float,
        c_int64, c_int64, c_int32, _pv, c_void_p]),
    'bb_mark4_encode': (c_int, [
        _pv, c_int32, _pv, _pi64, c_int64, c_int32, c_int32, c_int32,
        c_void_p]),
    'bb_mark4_encode_typed': (c_int, [
        _pv, c_int32, _pv, _pi64, c_int64, c_int32, c_int32, c_int32,
        c_void_p]),
    'bb_mark4_decode_words': (c_int, [
        _pv, c_int64, c_int32, c_int32, c_int32, _pf, _pv, c_void_p]),
    'bb_mark4_encode_words': (c_int, [
        _pv, c_int32, _pv, c_int64, c_int32, c_int32, c_int32, c_void_p]),
    'bb_decode_int8_transposed': (c_int, [
        _pv, _pi64, c_int64, c_int64, c_int64, c_int32, _pi64, _pi64, _pi64,
        _pv, c_void_p]),
    'bb_decode_int8_transposed_typed': (c_int, [
        _pv, _pi64, c_int64, c_int64, c_int64, c_int32, _pi64, _pi64, _pi64,
        c_int32, _pv, c_void_p]),
    'bb_encode_int8_transposed': (c_int, [
        _pv, c_int32, _pv, _pi64, c_int64, c_int64, c_int64, c_int32,
        c_void_p]),
    'bb_encode_int8_transposed_typed': (c_int, [
        _pv, c_int32, _pv, _pi64, c_int64, c_int64, c_int64, c_int32,
        c_void_p]),
    'bb_decode_int8_timefirst': (c_int, [
        _pv, _pi64, c_int64, c_int64, c_int32, c_int32, c_int32, _pi64,
        _pi64, _pi64, _pv, c_void_p]),
    'bb_decode_int8_timefirst_typed': (c_int, [
        _pv, _pi64, c_int64, c_int64, c_int32, c_int32, c_int32, _pi64,
        _pi64, _pi64, c_int32, _pv, c_void_p]),
    'bb_encode_int8_timefirst': (c_int, [
        _pv, c_int32, _pv, _pi64, c_int64, c_int64, c_int32, c_int32,
        c_int32, c_void_p]),
    'bb_encode_int8_timefirst_typed': (c_int, [
        _pv, c_int32, _pv, _pi64, c_int64, c_int64, c_int32, c_int32,
        c_int32, c_void_p]),
    'bb_vdif_scan': (c_int, [
        _pv, _pi64, c_int64, c_int64, c_int32, c_int32, c_int32, _pv, _pv,
        _pi64, _pv, c_int64, c_int32, c_int32, c_int32, c_void_p]),
    'bb_mark5b_scan': (c_int, [
        _pv, _pi64, c_int64, c_int64, _pv, _pi64, _pv, c_int64, c_int32,
        c_int32, c_int32, c_int32, c_void_p]),
    'bb_mark4_scan': (c_int, [
        _pv, _pi64, c_int64, c_int64, c_int32, c_int32, _pv, _pi64, _pv,
        c_int64, c_int32, c_int64, c_int64, c_void_p]),
    'bb_frames_assemble': (c_int, [
        _pv, c_int64, c_int64, c_int32, _pv, _pv, c_uint32, c_int64, c_int32,
        c_int64, _pi64, c_void_p]),
    'bb_host_copy': (c_int, [c_void_p, c_void_p, c_int64, c_int32]),
    'bb_host_copy_begin': (c_int, [c_void_p, c_void_p, c_int64, c_int32]),
    'bb_host_copy_wait': (c_int, [POINTER(c_int64)]),
    'bb_host_pread': (c_int, [c_int32, c_void_p, c_int64, c_int64, c_int32,
                              POINTER(c_int64)]),
    'bb_locate_frames': (c_int, [
        _pv, c_int64, c_int64, _pv, _pv, c_int32, c_int64, c_int64, c_int32,
        c_int32, c_int64, _pi64, c_int32, _pv, _pi64, c_int32, _pv,
        c_void_p]),
    'bb_index_table_init': (c_int, [_pv, c_int64, c_void_p]),
    'bb_vdif_index': (c_int, [
        _pv, c_int64, _pi64, _pv, c_int32, _pv, c_int32, c_int32, c_int32,
        c_int32, c_int32, c_int64, _pv, _pv, c_void_p]),
    'bb_mark5b_index': (c_int, [
        _pv, c_int64, _pi64, _pv, c_int32, c_int32, c_int32, c_int32,
        c_int32, c_int64, _pv, _pv, c_void_p]),
    'bb_mark4_index': (c_int, [
        _pv, c_int64, _pi64, _pv, c_int32, c_int32, c_int32, c_int32,
        c_int32, c_int32, c_int32, c_int64, c_int64, c_int32, c_int64, _pv,
        _pv, c_void_p]),
    'bb_index_table_finish': (c_int, [_pv, c_int64, _pi64, c_void_p]),
    'bb_state_counts': (c_int, [
        _pv, _pi64, c_int64, c_int32, c_int64, c_int32, c_int32, c_int64,
        c_int64, _pv, c_int64, c_void_p]),
    'bb_mark4_state_counts': (c_int, [
        _pv, _pi64, c_int64, c_int32, c_int32, c_int32, c_int64, c_int64,
        _pv, c_int64, c_void_p]),
    'bb_int8_moments': (c_int, [
        _pv, _pi64, c_int64, c_int32, c_int64, c_int32, c_int64, c_int64,
        _pv, c_int64, c_void_p]),
    'bb_probe_fill': (c_int, [_pv, c_int64, c_int32, c_void_p]),
    'bb_probe_copy': (c_int, [_pv, _pv, c_int64, c_void_p]),
    'bb_probe_expand': (c_int, [_pv, c_int64, _pv, c_int32, c_void_p]),
    'bb_probe_prefetch': (c_int, [_pv, c_int64, c_void_p]),
    'bb_probe_read': (c_int, [_pv, c_int64, c_void_p]),
}

# every symbol include/baseband_b200.h declares
EXPORTS = tuple(SIGNATURES)
# the reduced-precision decoders and encoders: bound when present, asked for
# by name when a float16 / bfloat16 result or input is handled
# (`kernels._typed`, `kernels._typed_encoder`)
OPTIONAL = ('bb_decode_bitfield_typed', 'bb_mark4_decode_typed',
            'bb_decode_int8_transposed_typed',
            'bb_decode_int8_timefirst_typed', 'bb_encode_bitfield_typed',
            'bb_mark4_encode_typed', 'bb_encode_int8_transposed_typed',
            'bb_encode_int8_timefirst_typed')


def bind(cdll, required=EXPORTS):
    """Attach argument/return types; raise if a required symbol is absent."""
    missing = []
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(cdll, name)
        except AttributeError:
            if name in required:
                missing.append(name)
            continue
        fn.restype = restype
        fn.argtypes = argtypes
    if missing:
        raise ImportError('library lacks symbols: ' + ', '.join(missing))
    return cdll


_lib = None


def load():
    """The CUDA library; built in-tree by ``python -m baseband_b200.build``."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                'baseband_b200: CUDA library not built ({}). Run '
                '`python -m baseband_b200.build` (needs nvcc); there is no '
                'CPU fallback.'.format(LIB_PATH))
        # Every symbol of include/baseband_b200.h must be there; a partial
        # library is a build error, not something to work around.
        _lib = bind(ctypes.CDLL(LIB_PATH),
                    required=() if os.environ.get('BB_ALLOW_PARTIAL') else
                    tuple(n for n in EXPORTS if n not in OPTIONAL))
        if _lib.bb_abi_version() != 2:
            raise ImportError('baseband_b200: ABI version mismatch')
    return _lib


_host = None


def host_io():
    """The library's host-side entry points (bb_host_copy, bb_host_pread):
    plain C++ threads, usable without a GPU."""
    global _host
    if _host is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError('baseband_b200: library not built ({})'
                              .format(LIB_PATH))
        _host = bind(ctypes.CDLL(LIB_PATH),
                     required=('bb_host_copy', 'bb_host_pread'))
    return _host


class BasebandCudaError(RuntimeError):
    pass


def check(status, lib=None):
    """Map a bb_status to the reference's exception types."""
    if status == BB_OK:
        return
    lib = lib or load()
    msg = lib.bb_last_error().decode('utf-8', 'replace')
    if status in (BB_ERR_ARGUMENT, BB_ERR_ALIGNMENT):
        raise ValueError(msg)
    if status == BB_ERR_UNSUPPORTED:
        raise KeyError(msg)
    raise BasebandCudaError(msg)
