"""CPU emulation of the kernel bodies + launch planning against the oracle.

The per-thread bodies in baseband_b200/csrc/*.cuh are host/device code; here
they are compiled with g++ (tests/emu) and every item is run in a loop.  This
checks index arithmetic, edge paths and quantisers without a GPU; the same
cases run on the real kernels in tests/test_gpu_parity.py.
"""
import ctypes

import numpy as np
import pytest

from baseband_b200 import levels
from oracle import codec
import emu_build
from bitfield_cases import (DECODE_CASES, ENCODE_CASES, make_decode_case,
                            oracle_decode, make_encode_case, oracle_encode)


@pytest.fixture(scope='module')
def emu():
    return emu_build.load()


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


@pytest.mark.parametrize('case', DECODE_CASES, ids=lambda c: c['id'])
def test_decode_bitfield(emu, case):
    c = make_decode_case(case)
    want = oracle_decode(c)
    out = np.full(want.size + 8, np.float32(np.nan))
    base = out[(-out.ctypes.data // 4) % 4:][:want.size]   # 16-byte aligned
    assert base.ctypes.data % 16 == 0
    lv = c['levels']
    rc = emu.bb_decode_bitfield(
        _ptr(c['raw']), _ptr(c['unit_offset']), c['nset'], c['nthread'],
        c['payload_nbytes'], c['bps'], c['nelem'], int(c['complex']),
        c['codec'],
        lv.ctypes.data_as(ctypes.POINTER(ctypes.c_float)) if lv is not None
        else None, c['fill'], c['sample_start'], c['nsample'], _ptr(base),
        None)
    assert rc == 0, emu.bb_last_error()
    assert np.array_equal(base.view('u4'), want.ravel().view('u4'))


@pytest.mark.parametrize('case', ENCODE_CASES, ids=lambda c: c['id'])
def test_encode_bitfield(emu, case):
    c = make_encode_case(case)
    want = oracle_encode(c)
    dst = np.full(c['dst_nbytes'], 0xEE, np.uint8)
    rc = emu.bb_encode_bitfield(
        _ptr(c['data']), c['dtype_code'], _ptr(dst), _ptr(c['unit_offset']),
        c['nset'], c['nthread'], c['payload_nbytes'], c['bps'], c['nelem'],
        c['quantiser'], None)
    assert rc == 0, emu.bb_last_error()
    assert np.array_equal(dst, want)


def test_golden_encode_vectors(emu, codec_vectors):
    """The reference's own outputs on threshold-hugging inputs."""
    g = codec_vectors
    for tag, code in (('f32', 0), ('f64', 1)):
        vals = np.ascontiguousarray(g['enc_in_' + tag])
        finite = np.ascontiguousarray(g['enc_in_finite_' + tag])
        for quant, name, bpss, src in (
                (0, 'vdif_enc%d_', (1, 2, 4, 8), vals),
                (1, 'm5b_enc%d_', (1, 2), vals),
                (2, {4: 'gsb4_enc_', 8: 'int8_enc_'}, (4, 8), finite)):
            for bps in bpss:
                key = (name[bps] if isinstance(name, dict)
                       else name % bps) + tag
                want = g[key]
                dst = np.zeros(want.size, np.uint8)
                off = np.zeros(1, np.int64)
                rc = emu.bb_encode_bitfield(
                    _ptr(src), code, _ptr(dst), _ptr(off), 1, 1, dst.size,
                    bps, 1, quant, None)
                assert rc == 0, emu.bb_last_error()
                bad = np.nonzero(dst != want)[0]
                assert bad.size == 0, (key, bad[:5])


def test_golden_decode_vectors(emu, codec_vectors):
    g = codec_vectors
    words = np.ascontiguousarray(g['words32'])
    off = np.zeros(1, np.int64)
    for key, bps, codec_id, lv in (
            ('vdif_dec1', 1, 0, levels.offset_binary(1)),
            ('vdif_dec2', 2, 0, levels.offset_binary(2)),
            ('vdif_dec4', 4, 0, levels.offset_binary(4)),
            ('vdif_dec8', 8, 0, levels.offset_binary(8)),
            ('m5b_dec1', 1, 0, levels.mark5b(1)),
            ('m5b_dec2', 2, 0, levels.mark5b(2))):
        want = g[key]
        out = np.zeros(want.size + 4, np.float32)
        base = out[(-out.ctypes.data // 4) % 4:][:want.size]
        lv = np.ascontiguousarray(lv, np.float32)
        rc = emu.bb_decode_bitfield(
            _ptr(words), _ptr(off), 1, 1, words.nbytes, bps, 1, 0, codec_id,
            lv.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), 0.0, 0,
            want.size, _ptr(base), None)
        assert rc == 0, emu.bb_last_error()
        assert np.array_equal(base.view('u4'), want.view('u4')), key
    b = np.ascontiguousarray(g['bytes'])
    for key, bps in (('gsb4_dec', 4), ('int8_dec', 8)):
        want = g[key]
        out = np.zeros(want.size + 4, np.float32)
        base = out[(-out.ctypes.data // 4) % 4:][:want.size]
        rc = emu.bb_decode_bitfield(_ptr(b), _ptr(off), 1, 1, b.nbytes, bps,
                                    1, 0, 1, None, 0.0, 0, want.size,
                                    _ptr(base), None)
        assert rc == 0
        assert np.array_equal(base, want), key


# ------------------------------------------------------------------ Mark 4
from mark4_cases import MODES, FRAME_CASES, make_frames, oracle_frames  # noqa
from baseband_b200 import levels as _levels  # noqa

_FP = ctypes.POINTER(ctypes.c_float)


def _aligned_f32(n):
    buf = np.full(n + 8, np.float32(np.nan))
    return buf[(-buf.ctypes.data // 4) % 4:][:n]


@pytest.mark.parametrize('tag', sorted(MODES))
def test_mark4_words_golden(emu, codec_vectors, tag):
    """One-hot and random words against the reference decoders, and the
    reference encoders on threshold-hugging inputs."""
    g = codec_vectors
    nchan, fanout, ft = MODES[tag]
    words = np.ascontiguousarray(g['m4_words_' + tag])
    want = g['m4_dec_' + tag]
    out = _aligned_f32(want.size)
    lv = np.ascontiguousarray(_levels.sign_magnitude(), np.float32)
    rc = emu.bb_mark4_decode_words(_ptr(words), words.size, nchan, fanout,
                                   int(ft), lv.ctypes.data_as(_FP), _ptr(out),
                                   None)
    assert rc == 0
    assert np.array_equal(out.reshape(want.shape).view('u4'), want.view('u4'))
    for ftag, code in (('f32', 0), ('f64', 1)):
        vals = g['m4_enc_in_%s_%s' % (tag, ftag)]
        src = np.zeros(vals.size + 4, vals.dtype)
        sh = (-src.ctypes.data // vals.itemsize) % (16 // vals.itemsize)
        src = src[sh:sh + vals.size]
        src[:] = vals.ravel()
        wantw = g['m4_enc_%s_%s' % (tag, ftag)]
        got = np.zeros(wantw.size, np.uint8)
        nword = vals.shape[0] // fanout
        rc = emu.bb_mark4_encode_words(_ptr(src), code, _ptr(got), nword,
                                       nchan, fanout, int(ft), None)
        assert rc == 0
        assert np.array_equal(got, wantw), (tag, ftag)


@pytest.mark.parametrize('case', FRAME_CASES, ids=lambda c: c[0])
def test_mark4_frames(emu, case):
    cid, mode, nframe, invalid, start, count, fill = case
    c = make_frames(mode, nframe, invalid, cid)
    want = oracle_frames(c, fill, start, count)
    out = _aligned_f32(want.size)
    lv = np.ascontiguousarray(_levels.sign_magnitude(), np.float32)
    rc = emu.bb_mark4_decode(_ptr(c['raw']), _ptr(c['unit_offset']), nframe,
                             c['nchan'], c['fanout'], int(c['ft']),
                             lv.ctypes.data_as(_FP), fill, start,
                             want.shape[0], _ptr(out), None)
    assert rc == 0, emu.emu_mark4_error()
    assert np.array_equal(out.reshape(want.shape).view('u4'), want.view('u4'))
    # encode the full decoded frames back: payload words must be identical
    full = oracle_frames(c, 0.0, 0, None)
    src = _aligned_f32(full.size)
    src[:] = full.ravel()
    dst = c['raw'].copy()
    for f in range(nframe):
        if c['unit_offset'][f] >= 0:
            o = c['truth'][f]
            dst[o:o + c['payload_nbytes']] = 0
    rc = emu.bb_mark4_encode(_ptr(src), 0, _ptr(dst), _ptr(c['unit_offset']),
                             nframe, c['nchan'], c['fanout'], int(c['ft']),
                             None)
    assert rc == 0
    assert np.array_equal(dst, c['raw'])


def test_mark4_sample_file(emu, sample_outputs):
    from conftest import sample_bytes
    raw = sample_bytes('sample.m4')
    off0 = int(sample_outputs['sample_m4_offset0'])
    want = sample_outputs['sample_m4_data']
    nframe = want.shape[0] // 80000
    src = np.zeros(raw.size + 16, np.uint8)
    sh = (-src.ctypes.data - off0) % 8
    src = src[sh:sh + raw.size]
    src[:] = raw
    uo = (off0 + np.arange(nframe) * 160000 + 1280).astype(np.int64)
    out = _aligned_f32(want.size)
    lv = np.ascontiguousarray(_levels.sign_magnitude(), np.float32)
    rc = emu.bb_mark4_decode(_ptr(src), _ptr(uo), nframe, 8, 4, 0,
                             lv.ctypes.data_as(_FP), -7.0, 0, want.shape[0],
                             _ptr(out), None)
    assert rc == 0
    assert np.array_equal(out.reshape(want.shape), want)


# --------------------------------------------------------- int8 transposed
import int8_cases  # noqa: E402


@pytest.mark.parametrize('case', int8_cases.CASES, ids=lambda c: c[0])
def test_int8_transposed(emu, case):
    c = int8_cases.make_case(case)
    want = int8_cases.oracle_decode(c)
    out = _aligned_f32(want.size)
    rc = emu.bb_decode_int8_transposed(
        _ptr(c['raw']), _ptr(c['unit_offset']), c['nunit'], c['nrow'],
        c['ncol'], c['ib'], _ptr(c['col_begin']), _ptr(c['col_end']),
        _ptr(c['out_col0']), _ptr(out), None)
    assert rc == 0
    assert np.array_equal(out.reshape(want.shape), want, equal_nan=True)
    # encode whole units back (full windows) and compare the packed bytes
    full = dict(c, col_begin=np.zeros(c['nunit'], np.int64),
                col_end=np.full(c['nunit'], c['ncol'], np.int64),
                out_col0=np.arange(c['nunit'], dtype=np.int64) * c['ncol'],
                ncols_out=c['nunit'] * c['ncol'])
    data = int8_cases.oracle_decode(full, fill=0.0)
    for dtype, code in ((np.float32, 0), (np.float64, 1)):
        src = np.ascontiguousarray(data, dtype)
        dst = c['raw'].copy()
        for u in range(c['nunit']):
            if c['unit_offset'][u] >= 0:
                dst[c['truth'][u]:c['truth'][u] + c['unit_nbytes']] = 0
        rc = emu.bb_encode_int8_transposed(
            _ptr(src), code, _ptr(dst), _ptr(c['unit_offset']), c['nunit'],
            c['nrow'], c['ncol'], c['ib'], None)
        assert rc == 0
        assert np.array_equal(dst, c['raw'])


@pytest.mark.parametrize('case', int8_cases.TF_CASES, ids=lambda c: c[0])
def test_int8_timefirst(emu, case):
    c = int8_cases.make_tf_case(case)
    want = int8_cases.oracle_tf_decode(c)
    out = _aligned_f32(want.size)
    out[:] = np.nan
    rc = emu.bb_decode_int8_timefirst(
        _ptr(c['raw']), _ptr(c['unit_offset']), c['nunit'], c['nsample'],
        c['nchan'], c['npol'], c['ib'], _ptr(c['t_begin']), _ptr(c['t_end']),
        _ptr(c['out_t0']), _ptr(out), None)
    assert rc == 0
    assert np.array_equal(out.reshape(want.shape), want, equal_nan=True)
    full = dict(c, t_begin=np.zeros(c['nunit'], np.int64),
                t_end=np.full(c['nunit'], c['nsample'], np.int64),
                out_t0=np.arange(c['nunit'], dtype=np.int64) * c['nsample'],
                nout=c['nunit'] * c['nsample'])
    data = int8_cases.oracle_tf_decode(full, fill=0.0)
    for dtype, code in ((np.float32, 0), (np.float64, 1)):
        src = _aligned_f32(data.size * (2 if code else 1)).view(dtype)
        src[:] = data.ravel()
        dst = c['raw'].copy()
        for u in range(c['nunit']):
            if c['unit_offset'][u] >= 0:
                dst[c['truth'][u]:c['truth'][u] + c['unit_nbytes']] = 0
        rc = emu.bb_encode_int8_timefirst(
            _ptr(src), code, _ptr(dst), _ptr(c['unit_offset']), c['nunit'],
            c['nsample'], c['nchan'], c['npol'], c['ib'], None)
        assert rc == 0
        assert np.array_equal(dst, c['raw'])


def test_fuzz_int8_timefirst(emu):
    for case in int8_cases.tf_fuzz_cases(60, seed=78):
        test_int8_timefirst(emu, case)


def test_int8_guppi_sample(emu, sample_outputs):
    """sample_puppi.raw frames through the transpose path == reference
    GUPPIPayload.data (channels first)."""
    from conftest import sample_bytes
    from oracle import stream
    raw = sample_bytes('sample_puppi.raw')
    frames = stream.guppi_scan(raw)
    h = frames[0]
    nrow, ncol = h['nchan'], h['samples_per_frame'] * h['npol']
    uo = np.array([f['offset'] + f['header_nbytes'] for f in frames], np.int64)
    n = len(frames)
    cb = np.zeros(n, np.int64)
    ce = np.full(n, ncol, np.int64)
    oc0 = np.arange(n, dtype=np.int64) * ncol
    want = sample_outputs['sample_puppi_frames']      # (n, spf, npol, nchan)
    out = _aligned_f32(want.size * 2)
    rc = emu.bb_decode_int8_transposed(_ptr(raw), _ptr(uo), n, nrow, ncol, 2,
                                       _ptr(cb), _ptr(ce), _ptr(oc0),
                                       _ptr(out), None)
    assert rc == 0
    got = out.view(np.complex64).reshape(want.shape)
    assert np.array_equal(got, want)


def test_int8_mkbf_sample(emu, sample_outputs):
    from conftest import sample_bytes
    from oracle import stream
    raw = sample_bytes('sample_mkbf.dada')
    h = stream.dada_parse_header(raw)
    want = sample_outputs['sample_mkbf_dada_data']     # (nsample, npol, nchan)
    nheap = want.shape[0] // 256
    nrow = h['npol'] * h['nchan']
    heap_nbytes = nrow * 256 * 2
    uo = (h['header_nbytes'] + np.arange(nheap) * heap_nbytes).astype(np.int64)
    cb = np.zeros(nheap, np.int64)
    ce = np.full(nheap, 256, np.int64)
    oc0 = np.arange(nheap, dtype=np.int64) * 256
    out = _aligned_f32(want.size * 2)
    rc = emu.bb_decode_int8_transposed(_ptr(raw), _ptr(uo), nheap, nrow, 256,
                                       2, _ptr(cb), _ptr(ce), _ptr(oc0),
                                       _ptr(out), None)
    assert rc == 0
    assert np.array_equal(out.view(np.complex64).reshape(want.shape), want)


def test_quant2_folded_thresholds(emu):
    """The 2-bit quantiser compares v with pre-folded thresholds; check it
    against the literal clip/add/floor-divide chain: every 1021st float32 of
    either sign plus +-200000 ulp around each threshold / clip bound, and
    +-200000 ulp around each for float64."""
    emu.emu_quant2_check.restype = ctypes.c_longlong
    emu.emu_quant2_check.argtypes = [ctypes.c_int, ctypes.c_int]
    assert emu.emu_quant2_check(0, 200000) == 0
    assert emu.emu_quant2_check(1, 200000) == 0


def test_affine8_is_the_8bit_table(emu):
    """The table-free 8-bit decode (byte permute, subtract, two-term
    reciprocal) reproduces the reference's 256 levels bit for bit, so the
    planner takes it for the standard table -- and not for another one."""
    emu.emu_affine8_mismatches.restype = ctypes.c_int
    emu.emu_affine8_mismatches.argtypes = [ctypes.c_void_p]
    table = np.ascontiguousarray(levels.offset_binary(8))
    assert emu.emu_affine8_mismatches(_ptr(table)) == 0
    other = table.copy()
    other[17] = np.nextafter(other[17], np.float32(1))
    assert emu.emu_affine8_mismatches(_ptr(other)) == 1001


def test_fuzz_bitfield(emu):
    """Random geometries through the planner + kernel bodies vs the oracle."""
    from bitfield_cases import fuzz_cases
    dec, enc = fuzz_cases(120, seed=20260101)
    for case in dec:
        test_decode_bitfield(emu, case)
    for case in enc:
        test_encode_bitfield(emu, case)


def test_matrix_bitfield(emu):
    """The multi-CTA coverage matrix through the kernel bodies vs the
    oracle (the GPU runs the same cases in test_gpu_bitfield)."""
    from bitfield_cases import matrix_cases
    dec, enc = matrix_cases()
    for case in dec:
        test_decode_bitfield(emu, case)
    for case in enc:
        test_encode_bitfield(emu, case)


def _planner_cells(emu):
    """Every (decode, encode) cell the default planner produces over a grid
    of geometries: bps, thread counts, elements per sample, two payload
    sizes (one with a number of words that is not a multiple of four), full
    reads, reads inside frames and unaligned reads."""
    from bitfield_cases import (DECODERS, QUANTISERS, plan_decode,
                                plan_encode)
    dec, enc = set(), set()
    for bps in (1, 2, 4, 8):
        for nthread in list(range(1, 10)) + [12, 16, 32, 64]:
            for nelem in (1, 2, 3, 4, 6, 8, 16, 32, 2048):
                bits = bps * nelem
                unit = bits * 32 // np.gcd(bits, 32) // 8    # bytes
                for payload in (unit * 8, unit * 9):
                    spf = payload * 8 // bits
                    total = 3 * spf
                    for start, count in ((0, total), (spf // 2, 2 * spf),
                                         (4, total - 8), (1, total - 2)):
                        mode, sel = plan_decode(
                            emu, 3, nthread, payload, bps, nelem, start,
                            count)[:2]
                        dec.update((mode, sel, bps, d) for d in DECODERS[bps])
                    mode = plan_encode(emu, 3, nthread, payload, bps,
                                       nelem)[0]
                    enc.update((mode, bps, q, t) for q in QUANTISERS[bps]
                               for t in ('f4', 'f8'))
    return dec, enc


def test_matrix_covers_every_planner_cell(emu):
    """matrix_cases() reaches exactly the kernel instances the planner can
    choose, and every case lands in the cell it is labelled with: a new mode
    or instance without a case, or a case that no longer plans where it
    says, fails here."""
    from bitfield_cases import matrix_cases, decode_cell, encode_cell
    want_dec, want_enc = _planner_cells(emu)
    dec, enc = matrix_cases()
    for c in dec:
        assert decode_cell(emu, c) == c['cell'], c['id']
    for c in enc:
        assert encode_cell(emu, c) == c['cell'], c['id']
    assert {c['cell'] for c in dec} == want_dec
    assert {c['cell'] for c in enc} == want_enc
    assert len({c['id'] for c in dec + enc}) == len(dec) + len(enc)
    # the variants of every decode cell: a full read; partial reads with
    # real fill, and complex fill where nelem is even, whose fill values
    # cover an ordinary number, -0.0 and NaN; for the modes that need
    # aligned reads, an unaligned read of the same bps and decoder that
    # falls back to another mode
    fills = {np.float32(f).view('u4').item() for f in (2.5, -0.0, np.nan)}
    for cell in want_dec:
        mine = [c for c in dec if c['cell'] == cell
                and 'fallback_of' not in c]
        assert any(c['start'] == 0 and c['count'] is None for c in mine)
        part = [c for c in mine if c['count'] is not None]
        assert any(not c['complex'] for c in part), cell
        if all(c['nelem'] % 2 == 0 for c in part):
            assert any(c['complex'] for c in part), cell
        assert {np.float32(c['fill']).view('u4').item()
                for c in part} >= fills, cell
        if cell[0] in ('WORDRUN', 'RUNS'):
            assert any(c.get('fallback_of') == cell[0]
                       and c['cell'][2:] == cell[2:] for c in dec), cell
    # and for every cell a case whose last CTA is partly filled down to its
    # last unrolled round (items counted by the real planner)
    from bitfield_cases import last_launch_items, last_round_partial
    tail = set()
    for c in dec + enc:
        if last_round_partial(last_launch_items(emu, c), c['cell'][0],
                              c['bps'], 'quant' in c):
            tail.add(c['cell'])
    assert tail == want_dec | want_enc


def test_matrix_case_sizes():
    """Each matrix case spans many CTAs and ends in a partly filled one: at
    least 4 MiB of float32 output (decode) or of input (encode), not a
    multiple of 64 KiB; the partial reads start and end inside frames."""
    from bitfield_cases import matrix_cases
    dec, enc = matrix_cases()
    for c in dec:
        spf = c['payload_nbytes'] * 8 // (c['bps'] * c['nelem'])
        count = c['count'] if c['count'] is not None else \
            c['nset'] * spf - c['start']
        nbytes = count * c['nthread'] * c['nelem'] * 4
        assert nbytes >= 4 << 20 and nbytes % (64 << 10), c['id']
        if c['start']:
            assert c['start'] % spf and (c['start'] + count) % spf, c['id']
            assert c['invalid'], c['id']
    for c in enc:
        spf = c['payload_nbytes'] * 8 // (c['bps'] * c['nelem'])
        nbytes = c['nset'] * spf * c['nthread'] * c['nelem'] * \
            np.dtype(c['dtype']).itemsize
        assert nbytes >= 4 << 20 and nbytes % (64 << 10), c['id']
        assert c['invalid'], c['id']


def test_fuzz_int8_transposed(emu):
    for case in int8_cases.fuzz_cases(60, seed=77):
        test_int8_transposed(emu, case)
