"""Shared case tables for the bit-field codec: used by the CPU emulation
tests and by the GPU parity tests, with the oracle as the checker."""
import ctypes
import zlib

import numpy as np

from baseband_b200 import levels
from oracle import codec


def _case(id, bps, nelem, nthread, nset, payload_nbytes, cplx=False,
          kind='vdif', start=0, count=None, invalid=(), shuffle=True,
          fill=0.0):
    return dict(id=id, bps=bps, nelem=nelem, nthread=nthread, nset=nset,
                payload_nbytes=payload_nbytes, complex=cplx, kind=kind,
                start=start, count=count, invalid=invalid, shuffle=shuffle,
                fill=fill)


DECODE_CASES = [
    # The section comments name the decomposition the planner picks for the
    # cases under them (`plan_decode` below tells).
    # ROWGROUP4: four single-channel threads per float4 (config C2; 2 bit
    # selects the levels in registers)
    _case('c2_2bit_16thr', 2, 1, 16, 3, 8000),
    _case('2bit_16thr_partial', 2, 1, 16, 3, 800, start=3217, count=4001),
    _case('2bit_16thr_invalid_partial', 2, 1, 16, 4, 404, start=1619,
          count=4200, invalid=(0, 17, 18, 35, 63), fill=-999.0),
    _case('2bit_16thr_odd_words', 2, 1, 16, 3, 36, invalid=(40,), fill=3.0),
    _case('8bit_12thr', 8, 1, 12, 2, 200, start=1, count=300),
    # ROWGROUP2: complex single channel / two channels, more than two (four)
    # threads
    _case('2bit_cplx_8thr', 2, 2, 8, 3, 260, cplx=True, start=77, count=700,
          invalid=(3, 12), fill=-5.0),
    _case('2bit_cplx_8thr_full', 2, 2, 8, 2, 800, cplx=True),
    _case('4bit_2chan_6thr', 4, 2, 6, 2, 96, start=7, count=150),
    # WORDROW4X2: rows of two float4 (8 single-channel threads, config C1)
    _case('c1_2bit_8thr', 2, 1, 8, 2, 5000),
    _case('2bit_8thr_invalid', 2, 1, 8, 3, 400, invalid=(1, 9, 10, 23),
          fill=-999.0),
    _case('1bit_8thr', 1, 1, 8, 2, 128, start=5, count=1999),
    # WORDROW2X2: rows of two float4 (4 threads of two elements)
    _case('1bit_2chan_4thr', 1, 2, 4, 2, 64),
    # WORDROW4 / WORDROW2: rows that are exactly one float4 (4 real / 2
    # complex threads)
    _case('2bit_4thr_one_sample', 2, 1, 4, 2, 64, start=255, count=2),
    _case('4bit_4thr', 4, 1, 4, 2, 256, invalid=(3,), fill=7.5),
    _case('1bit_4thr_rowrun', 1, 1, 4, 3, 68, start=33, count=1200,
          invalid=(6,), fill=-2.0),
    _case('8bit_4thr_rowrun', 8, 1, 4, 2, 404, start=3, count=700),
    _case('4bit_cplx_2thr_rowrun', 4, 2, 2, 3, 100, cplx=True, start=1,
          count=250, invalid=(3,), fill=5.0),
    _case('1bit_cplx_2thr_wordrow', 1, 2, 2, 3, 68, cplx=True, start=17,
          count=700, invalid=(4,), fill=-7.0),
    _case('2bit_cplx_2thr_wordrow', 2, 2, 2, 3, 200, cplx=True, start=399,
          count=403),
    _case('2bit_cplx_2thr', 2, 2, 2, 3, 512, cplx=True, invalid=(2,),
          fill=-3.0),
    _case('8bit_cplx_2thr_mwa', 8, 2, 2, 2, 1024, cplx=True, start=100,
          count=700),
    # WORDRUN: one thread, any nelem, reads aligned to float4
    _case('m5b_2bit_16ch', 2, 16, 1, 4, 10000, kind='mark5b',
          invalid=(2,), fill=-999.0),
    _case('m5b_2bit_8ch_partial', 2, 8, 1, 3, 10000, kind='mark5b',
          start=4999, count=7002),
    _case('m5b_1bit_4ch', 1, 4, 1, 2, 10000, kind='mark5b'),
    _case('2bit_1thr_1ch', 2, 1, 1, 3, 5000, start=4, count=59992),
    _case('2bit_1thr_3ch', 2, 3, 1, 2, 12 * 25),
    _case('1bit_16ch_bps1', 1, 16, 1, 2, 8000),
    _case('4bit_cplx_1024ch_aro', 4, 2048, 1, 2, 2048 * 5, cplx=True),
    # RUN: several threads, nelem a power of two >= 4 with more elements
    # than a word holds
    _case('8bit_2thr_cplx_4ch', 8, 8, 2, 2, 800, cplx=True, invalid=(0,),
          fill=-1.0),
    # RUNS: S = 2, 4, 8 samples per word, reads aligned to S rows (incl. one
    # that starts and ends inside frames), invalid units; and the same shapes
    # with an odd start, which must fall back to RUN
    _case('2bit_4thr_8ch', 2, 8, 4, 3, 640, invalid=(5,), fill=2.0,
          start=16, count=500),
    _case('4bit_3thr_4ch', 4, 4, 3, 2, 240),
    _case('runs_2bit_4thr_8ch_full', 2, 8, 4, 3, 640, invalid=(5, 6)),
    _case('runs_2bit_8thr_4ch_partial', 2, 4, 8, 3, 404, start=4 * 33,
          count=4 * 201, invalid=(11,), fill=-3.0),
    _case('runs_1bit_2thr_4ch', 1, 4, 2, 2, 68, start=8, count=8 * 30),
    _case('runs_4bit_5thr_4ch', 4, 4, 5, 2, 240, start=2, count=2 * 77,
          invalid=(0, 9)),
    _case('runs_2bit_2thr_cplx_2ch', 2, 4, 2, 2, 320, cplx=True, start=12,
          count=4 * 50, invalid=(1,), fill=5.0),
    _case('runs_2bit_4thr_8ch_s2_only', 2, 8, 4, 3, 640, start=2 * 15,
          count=2 * 401, invalid=(2,)),            # aligned to 2, not to 4
    _case('runs_8bit_3thr_4ch', 8, 4, 3, 2, 400, start=8, count=4 * 40,
          invalid=(4,), fill=1.5),                 # S = 1: four words an item
    _case('runs_2bit_2thr_16ch', 2, 16, 2, 2, 320, invalid=(3,)),
    _case('runs_4bit_2thr_8ch_cplx', 4, 8, 2, 2, 256, cplx=True, start=4,
          count=4 * 13),
    _case('run_2bit_8thr_4ch_odd_start', 2, 4, 8, 3, 404, start=4 * 33 + 1,
          count=4 * 201),
    # SCALAR: odd geometries / unaligned row ranges
    _case('2bit_3thr_1ch', 2, 1, 3, 3, 100, invalid=(4,), fill=9.0),
    _case('2bit_1thr_1ch_unaligned', 2, 1, 1, 2, 500, start=3, count=1001),
    _case('2bit_5thr_cplx', 2, 2, 5, 2, 200, cplx=True, invalid=(7,),
          fill=-999.0),
    _case('4bit_2thr_6ch', 4, 6, 2, 2, 240, start=1, count=77),
    _case('8bit_1thr_3ch_unaligned', 8, 3, 1, 2, 300, start=1, count=150),
    # non-standard level tables (always the shared-memory table path):
    # WORDROW4, WORDRUN, ROWGROUP4, ROWGROUP4 (2 bit), WORDROW2
    _case('custom8_4thr', 8, 1, 4, 2, 404, kind='custom', start=3, count=700),
    _case('custom8_1thr_cplx', 8, 2, 1, 2, 800, cplx=True, kind='custom'),
    _case('custom8_12thr', 8, 1, 12, 2, 200, kind='custom', invalid=(5,),
          fill=1.5),
    _case('custom2_16thr', 2, 1, 16, 2, 800, kind='custom'),
    _case('custom4_2thr_cplx', 4, 2, 2, 2, 100, cplx=True, kind='custom'),
    # signed-integer codecs: WORDRUN, WORDRUN, RUN, SCALAR
    _case('gsb_4bit_rawdump', 4, 1, 1, 2, 4096, kind='sint'),
    _case('dada_8bit_cplx_2pol', 8, 4, 1, 2, 6400, cplx=True, kind='sint'),
    _case('gsb_8bit_phased_2thr_cplx', 8, 1024, 2, 2, 4096, cplx=True,
          kind='sint', invalid=(1,), fill=0.5),
    _case('sint8_3thr', 8, 1, 3, 2, 120, kind='sint', start=5, count=100),
]


def custom_levels(bps):
    """A level table that is NOT the standard one (exercises the table path
    where the standard 8-bit levels are computed arithmetically)."""
    lv = np.ascontiguousarray(levels.offset_binary(bps), np.float32).copy()
    lv[::3] *= np.float32(1.25)
    lv[1] = np.float32(-77.0)
    return lv


def _levels(kind, bps):
    if kind == 'custom':
        return custom_levels(bps), 0
    if kind == 'vdif':
        return np.ascontiguousarray(levels.offset_binary(bps), np.float32), 0
    if kind == 'mark5b':
        return np.ascontiguousarray(levels.mark5b(bps), np.float32), 0
    return None, 1


def make_decode_case(case):
    rng = np.random.default_rng(zlib.crc32(case['id'].encode()))
    nunit = case['nset'] * case['nthread']
    nbytes = case['payload_nbytes']
    stride = nbytes + 32          # leave room for a (random) header
    order = rng.permutation(nunit) if case['shuffle'] else np.arange(nunit)
    raw = rng.integers(0, 256, nunit * stride + 64, dtype=np.uint8)
    unit_offset = (order * stride + 32).astype(np.int64)
    truth = unit_offset.copy()
    for u in case['invalid']:
        unit_offset[u] = -1
    spf = nbytes * 8 // (case['bps'] * case['nelem'])
    count = case['count']
    if count is None:
        count = case['nset'] * spf - case['start']
    lv, codec_id = _levels(case['kind'], case['bps'])
    return dict(case, raw=raw, unit_offset=unit_offset, truth=truth, spf=spf,
                sample_start=case['start'], nsample=count, levels=lv,
                codec=codec_id)


def _decode_unit(words, kind, bps):
    if kind == 'custom':
        codes = words.view(np.uint8)
        if bps < 8:
            shifts = np.arange(0, 8, bps, dtype=np.uint8)
            codes = (codes[:, None] >> shifts) & ((1 << bps) - 1)
        return custom_levels(bps)[codes.ravel()]
    if kind == 'vdif':
        return codec.vdif_decode(words, bps).ravel()
    if kind == 'mark5b':
        return codec.mark5b_decode(words, bps).ravel()
    b = words.view(np.int8)
    return (codec.gsb4_decode(b) if bps == 4 else codec.int8_decode(b)).ravel()


def oracle_decode(c):
    nset, nthread, nelem, spf = c['nset'], c['nthread'], c['nelem'], c['spf']
    full = np.empty((nset * spf, nthread, nelem), np.float32)
    for s in range(nset):
        for t in range(nthread):
            u = s * nthread + t
            blk = full[s * spf:(s + 1) * spf, t]
            if c['unit_offset'][u] < 0:
                blk[:] = c['fill']
                if c['complex']:
                    blk[:, 1::2] = 0.0
            else:
                o = c['truth'][u]
                words = c['raw'][o:o + c['payload_nbytes']].view('<u4')
                blk[:] = _decode_unit(words, c['kind'], c['bps']).reshape(
                    spf, nelem)
    return full[c['sample_start']:c['sample_start'] + c['nsample']]


def _ecase(id, bps, nelem, nthread, nset, payload_nbytes, quant='vdif',
           dtype='f4', invalid=(), offset0=32):
    return dict(id=id, bps=bps, nelem=nelem, nthread=nthread, nset=nset,
                payload_nbytes=payload_nbytes, quant=quant, dtype=dtype,
                invalid=invalid, offset0=offset0)


ENCODE_CASES = [
    _ecase('c2_2bit_16thr', 2, 1, 16, 3, 8000),
    _ecase('c2_2bit_16thr_f64', 2, 1, 16, 2, 800, dtype='f8'),
    _ecase('2bit_8thr_skip', 2, 1, 8, 3, 400, invalid=(1, 9)),
    _ecase('1bit_8thr', 1, 1, 8, 2, 128),
    _ecase('4bit_4thr', 4, 1, 4, 2, 256),
    _ecase('8bit_12thr', 8, 1, 12, 2, 200),
    _ecase('2bit_cplx_2thr', 2, 2, 2, 3, 512),
    _ecase('8bit_cplx_2thr_f64', 8, 2, 2, 2, 1024, dtype='f8'),
    _ecase('1bit_2chan_4thr', 1, 2, 4, 2, 64),
    _ecase('m5b_2bit_16ch', 2, 16, 1, 3, 10000, quant='mark5b'),
    _ecase('m5b_1bit_4ch_f64', 1, 4, 1, 2, 10000, quant='mark5b',
           dtype='f8'),
    _ecase('2bit_1thr_1ch', 2, 1, 1, 3, 5000),
    _ecase('2bit_1thr_3ch', 2, 3, 1, 2, 300),
    _ecase('4bit_cplx_1024ch', 4, 2048, 1, 2, 2048 * 5),
    _ecase('2bit_4thr_8ch', 2, 8, 4, 3, 640, invalid=(5,)),
    _ecase('4bit_3thr_4ch_f64', 4, 4, 3, 2, 240, dtype='f8'),
    _ecase('2bit_3thr_1ch', 2, 1, 3, 3, 100),
    _ecase('2bit_5thr_cplx', 2, 2, 5, 2, 200),
    _ecase('4bit_2thr_6ch', 4, 6, 2, 2, 240),
    # a row is one float4 (4 real / 2 complex threads): warp-cooperative
    # ROWWORD mode, chunks of 32 word positions crossing frame-set boundaries
    _ecase('1bit_4thr_rowword', 1, 1, 4, 3, 200),
    _ecase('2bit_4thr_rowword', 2, 1, 4, 3, 200, invalid=(2, 7)),
    _ecase('2bit_4thr_rowword_f64', 2, 1, 4, 2, 132, dtype='f8'),
    _ecase('8bit_4thr_rowword', 8, 1, 4, 3, 200),
    _ecase('1bit_cplx_2thr_rowword', 1, 2, 2, 3, 200),
    _ecase('4bit_cplx_2thr_rowword', 4, 2, 2, 3, 200, invalid=(0,)),
    _ecase('8bit_cplx_2thr_rowword', 8, 2, 2, 3, 200),
    _ecase('gsb_4bit', 4, 1, 1, 2, 4096, quant='sint'),
    _ecase('dada_8bit_cplx', 8, 4, 1, 2, 6400, quant='sint'),
    _ecase('gsb_8bit_2thr_f64', 8, 1024, 2, 2, 4096, quant='sint',
           dtype='f8'),
    # 8 bit in items of four words (RUNQ): one thread, or >= 16 elements per
    # thread row; payloads not at 16-byte offsets (four 4-byte stores); and
    # the shapes that must stay with one word per item
    _ecase('gsb_8bit_2thr', 8, 1024, 2, 3, 8192, quant='sint', invalid=(3,)),
    _ecase('vdif_8bit_1thr', 8, 1, 1, 3, 8000),
    _ecase('vdif_8bit_1thr_16ch_off8', 8, 16, 1, 3, 8000, offset0=40),
    _ecase('vdif_8bit_3thr_32ch_off4', 8, 32, 3, 2, 4096, offset0=36,
           invalid=(4,)),
    _ecase('dada_8bit_cplx_f64_off8', 8, 4, 1, 2, 6400, quant='sint',
           dtype='f8', offset0=8),
    _ecase('8bit_1thr_odd_words', 8, 2, 1, 2, 8008),
    _ecase('8bit_2thr_8ch', 8, 8, 2, 2, 4096),
]

_QUANT = {'vdif': 0, 'mark5b': 1, 'sint': 2}


def make_encode_case(case):
    rng = np.random.default_rng(zlib.crc32(case['id'].encode()))
    nset, nthread, nelem = case['nset'], case['nthread'], case['nelem']
    nbytes = case['payload_nbytes']
    spf = nbytes * 8 // (case['bps'] * nelem)
    scale = 40.0 if case['bps'] == 8 and case['quant'] == 'sint' else 2.5
    dtype = np.dtype(case['dtype'])
    data = (rng.standard_normal((nset * spf, nthread, nelem)) * scale
            ).astype(dtype)
    # sprinkle exact thresholds and half-integers
    flat = data.reshape(-1)
    marks = np.array([0.0, -0.0, 2.174564, -2.174564, 0.5, 1.5, 2.5, -0.5,
                      3.2618460000000002, 1e30, -1e30], dtype)
    flat[rng.integers(0, flat.size, marks.size * 4)] = np.tile(marks, 4)
    if case.get('specials'):
        # non-finite values, subnormals and signed zeros, many times over
        tiny = np.finfo(dtype).smallest_subnormal
        marks = np.concatenate([marks, np.array(
            [np.inf, -np.inf, np.nan, -np.nan, tiny, -tiny, 7 * tiny,
             -np.finfo(dtype).tiny / 2, -0.0], dtype)])
        flat[rng.integers(0, flat.size, marks.size * 64)] = np.tile(marks, 64)
    nunit = nset * nthread
    stride = nbytes + 32
    order = rng.permutation(nunit)
    unit_offset = (order * stride + case.get('offset0', 32)).astype(np.int64)
    truth = unit_offset.copy()
    for u in case['invalid']:
        unit_offset[u] = -1
    # 16-byte aligned input
    buf = np.zeros(data.size + 4, dtype)
    shift = (-buf.ctypes.data // dtype.itemsize) % (16 // dtype.itemsize)
    aligned = buf[shift:shift + data.size]
    aligned[:] = flat
    return dict(case, data=aligned, shaped=aligned.reshape(data.shape),
                unit_offset=unit_offset, truth=truth, spf=spf,
                dst_nbytes=nunit * stride + 64,
                dtype_code=0 if dtype.itemsize == 4 else 1,
                quantiser=_QUANT[case['quant']])


def oracle_encode(c):
    dst = np.full(c['dst_nbytes'], 0xEE, np.uint8)
    spf, nthread = c['spf'], c['nthread']
    for s in range(c['nset']):
        for t in range(nthread):
            u = s * nthread + t
            if c['unit_offset'][u] < 0:
                continue
            vals = np.ascontiguousarray(
                c['shaped'][s * spf:(s + 1) * spf, t]).ravel()
            with np.errstate(all='ignore'):
                if c['quant'] == 'vdif':
                    enc = codec.vdif_encode(vals.copy(), c['bps'])
                elif c['quant'] == 'mark5b':
                    enc = codec.mark5b_encode(vals.copy(), c['bps'])
                elif c['bps'] == 4:
                    enc = codec.gsb4_encode(vals)
                else:
                    enc = codec.int8_encode(vals)
            o = c['truth'][u]
            dst[o:o + c['payload_nbytes']] = np.ascontiguousarray(
                enc).ravel().view(np.uint8)
    return dst


def fuzz_cases(n, seed):
    """Seeded random decode / encode geometries covering every mode of the
    planner (thread counts 1-9, 1-16 elements, odd payload sizes, partial
    sample ranges, invalid units, all codecs)."""
    rng = np.random.default_rng(seed)
    dec, enc = [], []
    for i in range(n):
        kind = rng.choice(['vdif', 'vdif', 'mark5b', 'sint'])
        bps = int(rng.choice({'vdif': [1, 2, 4, 8], 'mark5b': [1, 2],
                              'sint': [4, 8]}[kind]))
        nthread = int(rng.choice([1, 1, 2, 2, 3, 4, 4, 5, 8, 9]))
        nelem = int(rng.choice([1, 1, 2, 2, 3, 4, 8, 16]))
        cplx = bool(nelem % 2 == 0 and rng.random() < 0.4)
        nset = int(rng.integers(1, 4))
        # payload: whole 32-bit words holding whole samples
        bits = bps * nelem
        unit = bits * 32 // np.gcd(bits, 32)          # lcm(bits, 32) bits
        payload = int(unit // 8 * rng.integers(1, 40))
        spf = payload * 8 // bits
        total = nset * spf
        if rng.random() < 0.5:
            start = int(rng.integers(0, total))
            count = int(rng.integers(1, total - start + 1))
        else:
            start, count = 0, None
        ninv = int(rng.integers(0, 3))
        invalid = tuple(int(v) for v in rng.choice(
            nset * nthread, size=min(ninv, nset * nthread), replace=False))
        fill = float(rng.choice([0.0, -999.0, 2.5]))
        cid = 'fuzz%d_%s_b%d_t%d_e%d' % (i, kind, bps, nthread, nelem)
        dec.append(_case(cid, bps, nelem, nthread, nset, payload, cplx=cplx,
                         kind=kind, start=start, count=count,
                         invalid=invalid, fill=fill))
        quant = {'vdif': 'vdif', 'mark5b': 'mark5b', 'sint': 'sint'}[kind]
        enc.append(_ecase(cid, bps, nelem, nthread, nset, payload,
                          quant=quant, invalid=invalid,
                          dtype='f8' if rng.random() < 0.3 else 'f4'))
    return dec, enc


# ---------------------------------------------------------------------------
# Planner cells.  Every decomposition the planner picks runs as its own
# kernel instance per bps and decoder (decode) or per bps, quantiser and input
# type (encode): a "cell".  `matrix_cases` holds multi-CTA cases for every
# cell the default planner produces; test_emulation checks that the set is
# complete and that each case lands in the cell it is labelled with.
MODE_NAMES = {0: 'ROWGROUP4', 1: 'ROWGROUP2', 2: 'RUN', 3: 'SCALAR',
              4: 'WORDRUN', 7: 'WORDROW4', 8: 'ROWWORD4', 9: 'ROWWORD2',
              10: 'WORDROW2', 11: 'WORDROW4X2', 12: 'WORDROW2X2',
              13: 'TILE4', 14: 'TILE2', 15: 'RUNS', 16: 'RUNQ'}
# decoder instances per bps: 'levels' at 8 bit is a table other than the
# standard one (the standard one is computed: 'affine8')
DECODERS = {1: ('levels',), 2: ('levels',), 4: ('levels', 'sint'),
            8: ('affine8', 'levels', 'sint')}
QUANTISERS = {1: ('vdif', 'mark5b'), 2: ('vdif', 'mark5b'),
              4: ('vdif', 'sint'), 8: ('vdif', 'sint')}


def _plan_result(emu, rc, info):
    if rc:
        raise ValueError(emu.bb_last_error())
    return (MODE_NAMES[info[0]],) + tuple(int(v) for v in info[1:])


def plan_decode(emu, nset, nthread, payload_nbytes, bps, nelem,
                sample_start, nsample, cplx=False):
    """(mode, sel, number of launches, frame sets of the first launch,
    items of the last launch) of the real planner for a decode call; `emu`
    is the emulation library."""
    info = (ctypes.c_int64 * 5)()
    rc = emu.emu_plan_decode(
        ctypes.c_int64(nset), ctypes.c_int32(nthread),
        ctypes.c_int64(payload_nbytes), ctypes.c_int32(bps),
        ctypes.c_int32(nelem), ctypes.c_int32(int(cplx)),
        ctypes.c_int64(sample_start), ctypes.c_int64(nsample), info)
    return _plan_result(emu, rc, info)


def plan_encode(emu, nset, nthread, payload_nbytes, bps, nelem):
    """As plan_decode, for an encode call."""
    info = (ctypes.c_int64 * 5)()
    rc = emu.emu_plan_encode(
        ctypes.c_int64(nset), ctypes.c_int32(nthread),
        ctypes.c_int64(payload_nbytes), ctypes.c_int32(bps),
        ctypes.c_int32(nelem), info)
    return _plan_result(emu, rc, info)


def decoder_of(kind, bps):
    if kind == 'sint':
        return 'sint'
    return 'affine8' if bps == 8 and kind != 'custom' else 'levels'


def _plan_case(emu, case):
    if 'quant' in case:
        return plan_encode(emu, case['nset'], case['nthread'],
                           case['payload_nbytes'], case['bps'], case['nelem'])
    spf = case['payload_nbytes'] * 8 // (case['bps'] * case['nelem'])
    count = case['count']
    if count is None:
        count = case['nset'] * spf - case['start']
    return plan_decode(emu, case['nset'], case['nthread'],
                       case['payload_nbytes'], case['bps'], case['nelem'],
                       case['start'], count, case['complex'])


def last_launch_items(emu, case):
    """Items of the last launch the planner makes of a matrix case."""
    return _plan_case(emu, case)[4]


def decode_cell(emu, case):
    mode, sel = _plan_case(emu, case)[:2]
    return mode, sel, case['bps'], decoder_of(case['kind'], case['bps'])


def encode_cell(emu, case):
    mode = _plan_case(emu, case)[0]
    return mode, case['bps'], case['quant'], case['dtype']


_MIN_BYTES = 4 << 20            # output (decode) / input (encode) per case
_SET_FLOATS = 300000            # about this many values per frame set


def _payload(bps, nelem, rowlen):
    """Whole words of whole samples, spf a multiple of 8, roughly
    _SET_FLOATS values per frame set, not a power of two."""
    bits = bps * nelem
    unit = bits * 32 // np.gcd(bits, 32)          # lcm(bits, 32) bits
    spf_unit = unit // bits
    m = max(1, round(_SET_FLOATS / (rowlen * spf_unit * 8))) | 1
    return unit // 8 * 8 * m


def _nset(set_values, itemsize, margin):
    n = -(-_MIN_BYTES // (set_values * itemsize)) + margin
    while (n * set_values * itemsize) % (64 << 10) == 0:
        n += 1
    return n


def _invalid(nthread, first_set, last_set):
    """The first and last unit touched and a few in the middle."""
    mid = (first_set + last_set) // 2
    units = {first_set * nthread, last_set * nthread + nthread - 1,
             mid * nthread + nthread // 2, (mid + 1) * nthread + nthread - 1,
             (mid + 1) * nthread}
    return tuple(sorted(units))


# Items per CTA of each kernel instance: kBlock (256) threads times the
# unroll factor (Unroll / EncUnroll in bb_bitfield.cu, restated).
def cta_items(mode, bps, encode=False):
    if encode:
        if mode in ('ROWGROUP4', 'ROWGROUP2'):
            f4 = (32 if mode == 'ROWGROUP4' else 16) // bps
        elif mode in ('ROWWORD4', 'ROWWORD2'):
            f4 = (32 if mode == 'ROWWORD4' else 16) // bps
        else:
            return 256 * 4
        return 256 * (1 if f4 >= 16 else 16 // f4)
    f4 = {'ROWGROUP4': min(32 // bps, 8), 'ROWGROUP2': min(16 // bps, 8),
          'WORDRUN': 8 // bps, 'WORDROW4': 32 // bps, 'WORDROW2': 16 // bps,
          'WORDROW4X2': 64 // bps, 'WORDROW2X2': 32 // bps,
          'RUNS': 4}.get(mode, 1)
    target = 8 if (mode in ('WORDRUN', 'WORDROW4', 'ROWGROUP4', 'ROWGROUP2')
                   or mode == 'WORDROW2' and bps <= 2) else 16
    return 256 * (1 if f4 >= target else target // f4)


def last_round_partial(nitems, mode, bps, encode=False):
    """The grid's last CTA is partly filled and its last unrolled round
    holds some items but not all."""
    span = cta_items(mode, bps, encode)
    return span - 256 < nitems % span < span


def _full_items(mode, bps, nthread, nelem, payload, nset, encode=False):
    """Items of a one-launch full-range call (the planner's arithmetic)."""
    nword = payload // 4
    spf = payload * 8 // (bps * nelem)
    rowlen = nthread * nelem
    if mode in ('ROWGROUP4', 'ROWGROUP2'):
        g = 4 if mode == 'ROWGROUP4' else 2
        tpw = 32 // bps // (4 // g)
        split = 1 if encode or tpw <= 8 else tpw // 8
        return nword * (nthread // g) * split * nset
    if mode in ('WORDRUN', 'ROWWORD4', 'ROWWORD2') or mode.startswith(
            'WORDROW'):
        return -(-nword * nset // 32) * 32
    if encode:
        return (nword // 4 if mode == 'RUNQ' else nword) * nthread * nset
    if mode == 'RUN':
        return spf * rowlen // 4 * nset
    if mode == 'RUNS':
        return spf // max(32 // (bps * nelem), 4) * rowlen // 4 * nset
    return spf * rowlen * nset


def _tail_shape(mode, bps, nthread, nelem, payload, nset, encode=False):
    """(payload, nset), from the given ones on, of a full-range call that
    leaves the last unrolled round of the last CTA partly filled."""
    bits = bps * nelem
    step = bits * 32 // np.gcd(bits, 32) // 8     # whole words and samples
    if mode == 'RUNS':
        step *= 8                                     # spf % 8 == 0
    for p in range(payload, payload + 64 * step, step):
        for n in range(nset, nset + 64):
            items = _full_items(mode, bps, nthread, nelem, p, n, encode)
            size = n * (p * 8 // bits) * nthread * nelem
            if last_round_partial(items, mode, bps, encode) and size % 16384:
                return p, n
    return payload, nset


_DEC_KIND = {'levels': 'vdif', 'affine8': 'vdif', 'sint': 'sint'}


def _dec_shape(mode, bps, variant):
    cpw = 32 // bps
    if mode == 'ROWGROUP4':     # 16- and 12-thread single-channel VDIF
        return (16 if variant == 0 else 12), 1
    return {'ROWGROUP2': (8, 2), 'WORDROW4': (4, 1), 'WORDROW2': (2, 2),
            'WORDROW4X2': (8, 1), 'WORDROW2X2': (4, 2),
            'WORDRUN': (1, 16 if bps <= 2 else 4), 'RUNS': (3, 4),
            'RUN': (2, 2 * cpw),
            'SCALAR': (3, 1) if bps <= 2 else (5, 2)}[mode]


def _read_align(mode, nelem, tpw):
    if mode == 'WORDRUN':                 # float4-aligned rows
        return 4 // int(np.gcd(nelem, 4))
    if mode == 'RUNS':                    # groups of max(S, 4) rows
        return max(tpw, 4)
    return 1


def _decode_matrix():
    cases = []
    fills = (2.5, -0.0, float('nan'))
    for mode in ('ROWGROUP4', 'WORDROW4X2', 'ROWGROUP2', 'WORDROW4',
                 'WORDROW2', 'WORDROW2X2', 'WORDRUN', 'RUNS', 'RUN',
                 'SCALAR'):
        for bps in (1, 4, 2, 8):
            for dec in DECODERS[bps]:
                sel = int(mode == 'ROWGROUP4' and bps == 2)
                cell = (mode, sel, bps, dec)
                kind = 'custom' if (dec == 'levels' and bps == 8) else \
                    _DEC_KIND[dec]
                if kind == 'vdif' and mode == 'WORDRUN' and bps <= 2:
                    kind = 'mark5b'
                for v in range(4):
                    nthread, nelem = _dec_shape(mode, bps, v)
                    rowlen = nthread * nelem
                    payload = _payload(bps, nelem, rowlen)
                    spf = payload * 8 // (bps * nelem)
                    nset = _nset(spf * rowlen, 4, 2)
                    cid = 'm_%s_%s_b%d_%dx%d_v%d' % (
                        mode.lower(), dec, bps, nthread, nelem, v)
                    if v == 0:              # (a) full range, all valid
                        payload, nset = _tail_shape(mode, bps, nthread,
                                                    nelem, payload, nset)
                        cases.append(dict(_case(
                            cid, bps, nelem, nthread, nset, payload,
                            kind=kind), cell=cell))
                        continue
                    # (b) from inside a frame (inside a word where the mode
                    # allows) to inside a frame, invalid units at both ends
                    tpw = 32 // (bps * nelem)
                    al = _read_align(mode, nelem, tpw)
                    start = (spf // 3 // al + v) * al
                    end = ((nset - 1) * spf + 2 * spf // 3) // al * al
                    if al < tpw:
                        start += al if start % tpw == 0 else 0
                        end += al if end % tpw == 0 else 0
                    while ((end - start) * rowlen) % 16384 == 0:
                        end -= al
                    cplx = nelem % 2 == 0 and v == 2
                    cases.append(dict(_case(
                        cid, bps, nelem, nthread, nset, payload, cplx=cplx,
                        kind=kind, start=start, count=end - start,
                        invalid=_invalid(nthread, start // spf,
                                         (end - 1) // spf),
                        fill=fills[v - 1]), cell=cell))
                # reads that are not aligned as the mode needs fall back
                if mode in ('WORDRUN', 'RUNS'):
                    nthread, nelem = (1, 1) if mode == 'WORDRUN' else (3, 4)
                    rowlen = nthread * nelem
                    payload = _payload(bps, nelem, rowlen)
                    spf = payload * 8 // (bps * nelem)
                    nset = _nset(spf * rowlen, 4, 2)
                    start, end = spf // 2 + 1, nset * spf - spf // 2 - 2
                    while ((end - start) * rowlen) % 16384 == 0:
                        end -= 1
                    cid = 'm_%s_unaligned_%s_b%d' % (mode.lower(), dec, bps)
                    cases.append(dict(_case(
                        cid, bps, nelem, nthread, nset, payload, kind=kind,
                        start=start, count=end - start,
                        invalid=_invalid(nthread, start // spf,
                                         (end - 1) // spf), fill=-7.0),
                        cell=('SCALAR' if mode == 'WORDRUN' else 'RUN', 0,
                              bps, dec), fallback_of=mode))
    return cases


def _enc_shape(mode, bps):
    return {'ROWGROUP4': (16, 1), 'ROWGROUP2': (8, 2), 'ROWWORD4': (4, 1),
            'ROWWORD2': (2, 2), 'RUN': (1, 16) if bps <= 4 else (3, 4),
            'RUNQ': (1, 4),
            'SCALAR': (3, 1) if bps <= 2 else (5, 2)}[mode]


def _encode_matrix():
    cases = []
    for mode in ('ROWGROUP4', 'ROWWORD4', 'ROWGROUP2', 'ROWWORD2', 'RUN',
                 'RUNQ', 'SCALAR'):
        for bps in (4, 1, 2, 8):
            if (mode == 'RUNQ' and bps != 8 or mode == 'ROWWORD4' and bps > 4
                    or mode == 'ROWWORD2' and bps > 2):
                continue
            for quant in QUANTISERS[bps]:
                for dtype in ('f4', 'f8'):
                    nthread, nelem = _enc_shape(mode, bps)
                    rowlen = nthread * nelem
                    payload = _payload(bps, nelem, rowlen)
                    spf = payload * 8 // (bps * nelem)
                    isz = np.dtype(dtype).itemsize
                    payload, nset = _tail_shape(
                        mode, bps, nthread, nelem, payload,
                        _nset(spf * rowlen, isz, 1), True)
                    cid = 'm_%s_%s_b%d_%s_%dx%d' % (mode.lower(), quant, bps,
                                                    dtype, nthread, nelem)
                    case = _ecase(cid, bps, nelem, nthread, nset, payload,
                                  quant=quant, dtype=dtype,
                                  invalid=_invalid(nthread, 0, nset - 1))
                    cases.append(dict(case, specials=True,
                                      cell=(mode, bps, quant, dtype)))
    return cases


def matrix_cases():
    """Multi-CTA decode and encode cases (each at least 4 MiB of float32
    output / of input, not a multiple of 64 KiB) for every cell of the
    planner: decode full ranges; partial ranges starting and ending inside
    frames with invalid units at both ends and in the middle (real and
    complex fill, fill values 2.5, -0.0 and NaN); unaligned reads that fall
    back from WORDRUN / RUNS; encode with invalid units and non-finite,
    subnormal and signed-zero inputs."""
    return _decode_matrix(), _encode_matrix()
