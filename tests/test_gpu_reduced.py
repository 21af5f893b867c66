"""float16 / bfloat16 decoder output on the GPU.  The rule: a reduced result
equals the float32 result converted with torch's ``.to(dtype)``, bit for
bit, -0.0 and +-inf included, NaN by position only.

ABI level: every decode cell of the planner, the Mark 4 and int8 case tables
and a partial read across a launch split, each into a view of a larger
buffer whose sentinels must stay untouched; output alignment and the
encoders' refusal of 16-bit input.  Public API: every format's streams
(tests/reduced_cases.py) with device and host output."""
import ctypes

import numpy as np
import pytest
import torch

from baseband_b200 import _lib, kernels, levels
import reduced_cases
from reduced_cases import HALF, assert_reduced
from bitfield_cases import (DECODE_CASES, make_decode_case, oracle_decode,
                            matrix_cases)

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
GUARD = 32768                       # 64 KiB of sentinel either side
SENTINEL = 0x7dad                   # a float16 / bfloat16 no decode makes


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _guarded(n, dtype):
    buf = torch.full((n + 2 * GUARD,), SENTINEL, dtype=torch.int16,
                     device=DEV)
    return buf, buf[GUARD:GUARD + n].view(dtype)


def _check_guard(buf):
    assert bool((buf[:GUARD] == SENTINEL).all())
    assert bool((buf[-GUARD:] == SENTINEL).all())


MATRIX_DECODE = matrix_cases()[0]


@pytest.mark.parametrize('case', DECODE_CASES + MATRIX_DECODE,
                         ids=lambda c: c['id'])
def test_decode_bitfield(case):
    c = make_decode_case(case)
    want = _t(oracle_decode(c))
    args = (_t(c['raw']), _t(c['unit_offset']), c['nset'], c['nthread'],
            c['payload_nbytes'], c['bps'], c['nelem'], c['complex'],
            c['codec'], c['levels'], c['fill'], c['sample_start'],
            c['nsample'])
    for dtype in HALF:
        buf, view = _guarded(want.numel(), dtype)
        out = kernels.decode_bitfield(*args, out=view.view(want.shape))
        assert out.data_ptr() == view.data_ptr() and out.dtype == dtype
        assert_reduced(out, want, dtype)
        _check_guard(buf)
        # allocated by the wrapper
        assert_reduced(kernels.decode_bitfield(*args, dtype=dtype), want,
                       dtype)


@pytest.mark.parametrize('case', __import__('mark4_cases').FRAME_CASES,
                         ids=lambda c: c[0])
def test_mark4_frames(case):
    from mark4_cases import make_frames, oracle_frames
    cid, mode, nframe, invalid, start, count, fill = case
    c = make_frames(mode, nframe, invalid, cid)
    want = _t(oracle_frames(c, fill, start, count))
    for dtype in HALF:
        buf, view = _guarded(want.numel(), dtype)
        kernels.mark4_decode(_t(c['raw']), _t(c['unit_offset']), nframe,
                             c['nchan'], c['fanout'], c['ft'],
                             levels.sign_magnitude(), fill, start,
                             want.shape[0], out=view)
        assert_reduced(view.view(want.shape), want, dtype)
        _check_guard(buf)


def _int8_cases():
    import int8_cases
    return ([('t', c) for c in int8_cases.CASES]
            + [('tf', c) for c in int8_cases.TF_CASES])


@pytest.mark.parametrize('kind,case', _int8_cases(),
                         ids=lambda c: c if isinstance(c, str) else c[0])
def test_int8(kind, case):
    import int8_cases
    c = int8_cases.make_case(case) if kind == 't' \
        else int8_cases.make_tf_case(case)
    want = _t(int8_cases.oracle_decode(c) if kind == 't'
              else int8_cases.oracle_tf_decode(c))
    nan = {torch.float16: 0x7e00, torch.bfloat16: 0x7fc0}
    for dtype in HALF:
        buf, view = _guarded(want.numel(), dtype)
        view.view(torch.int16).fill_(nan[dtype])   # untouched stays NaN
        if kind == 't':
            kernels.decode_int8_transposed(
                _t(c['raw']), _t(c['unit_offset']), c['nunit'], c['nrow'],
                c['ncol'], c['ib'], _t(c['col_begin']), _t(c['col_end']),
                _t(c['out_col0']), view)
        else:
            kernels.decode_int8_timefirst(
                _t(c['raw']), _t(c['unit_offset']), c['nunit'],
                c['nsample'], c['nchan'], c['npol'], c['ib'],
                _t(c['t_begin']), _t(c['t_end']), _t(c['out_t0']), view)
        assert_reduced(view.view(want.shape), want, dtype)
        _check_guard(buf)


def test_partial_read_across_launch_split():
    """8-bit single-thread WORDRUN just past one launch (test_gpu_large's
    geometry): invalid units on both sides of the split, a read from inside
    the first frame to inside the last."""
    import emu_build
    from bitfield_cases import plan_decode
    emu = emu_build.load()
    bps, nelem, payload, fill = 8, 1, 8000, -999.0
    nset = 0x3ffffff // (payload // 4) + 7
    start = (payload // 3) // 4 * 4 + 4
    end = ((nset - 1) * payload + 2 * payload // 3) // 4 * 4
    mode, _, nlaunch, split, _ = plan_decode(emu, nset, 1, payload, bps,
                                             nelem, start, end - start)
    assert (mode, nlaunch) == ('WORDRUN', 2)
    g = torch.Generator(device=DEV).manual_seed(78)
    raw = torch.randint(0, 256, (nset * (payload + 32),), dtype=torch.uint8,
                        device=DEV, generator=g)
    uo = torch.arange(nset, dtype=torch.int64, device=DEV) * (payload + 32) \
        + 32
    uo[[split - 1, split, nset - 1]] = -1
    args = (raw, uo, nset, 1, payload, bps, nelem, False,
            kernels.CODEC_LEVELS, levels.offset_binary(8), fill, start,
            end - start)
    want = kernels.decode_bitfield(*args)
    for dtype in HALF:
        buf, view = _guarded(want.numel(), dtype)
        kernels.decode_bitfield(*args, out=view)
        assert_reduced(view.view(want.shape), want, dtype)
        _check_guard(buf)
        del buf, view
    del want
    torch.cuda.empty_cache()


def test_out_alignment():
    """16-bit output needs 8-byte alignment (float32: 16); an 8-byte
    aligned view gets the same values."""
    c = make_decode_case(DECODE_CASES[0])
    want = _t(oracle_decode(c)).reshape(-1)
    args = (_t(c['raw']), _t(c['unit_offset']), c['nset'], c['nthread'],
            c['payload_nbytes'], c['bps'], c['nelem'], c['complex'],
            c['codec'], c['levels'], c['fill'], c['sample_start'],
            c['nsample'])
    for dtype in HALF:
        buf = torch.zeros(want.numel() + 8, dtype=dtype, device=DEV)
        assert buf.data_ptr() % 16 == 0
        with pytest.raises(ValueError):              # 4-byte aligned
            kernels.decode_bitfield(*args, out=buf[2:2 + want.numel()])
        view = buf[4:4 + want.numel()]               # 8-byte aligned
        kernels.decode_bitfield(*args, out=view)
        assert_reduced(view, want, dtype)
        with pytest.raises(TypeError):
            kernels.decode_bitfield(*args, out=torch.empty(
                want.numel(), dtype=torch.float64, device=DEV))


def test_encoders_refuse_16bit_input():
    lib = _lib.load()
    data = torch.zeros(4096, dtype=torch.float16, device=DEV)
    dst = torch.zeros(4096, dtype=torch.uint8, device=DEV)
    uo = torch.zeros(1, dtype=torch.int64, device=DEV)
    p = [ctypes.c_void_p(t.data_ptr()) for t in (data, dst, uo)]
    for code in (_lib.F16, _lib.BF16):
        assert lib.bb_encode_bitfield(p[0], code, p[1], p[2], 1, 1, 1024, 2,
                                      1, 0, None) == _lib.BB_ERR_ARGUMENT
        assert lib.bb_mark4_encode(p[0], code, p[1], p[2], 1, 8, 4, 0,
                                   None) == _lib.BB_ERR_ARGUMENT
        assert lib.bb_encode_int8_transposed(
            p[0], code, p[1], p[2], 1, 32, 64, 1,
            None) == _lib.BB_ERR_ARGUMENT
        assert lib.bb_encode_int8_timefirst(
            p[0], code, p[1], p[2], 1, 16, 8, 2, 2,
            None) == _lib.BB_ERR_ARGUMENT
    torch.cuda.synchronize()


# ------------------------------------------------------------ public API
@pytest.mark.parametrize('name', sorted(reduced_cases.STREAMS))
def test_stream_reads(name):
    reduced_cases.check_stream(name, DEV)


def test_out_variants():
    reduced_cases.check_out_variants(DEV, pinned=True)


def test_shapes_and_subsets():
    reduced_cases.check_shapes_and_subsets(DEV)


def test_small_reads_and_pickle():
    reduced_cases.check_small_reads_and_pickle()


def test_host_result_is_pinned():
    import baseband_b200 as bb
    from conftest import sample_path
    with bb.vdif.open(sample_path('sample.vdif'), 'rs',
                      dtype='float16') as fh:
        data = fh.read()
    assert data.dtype == torch.float16 and data.is_pinned()
