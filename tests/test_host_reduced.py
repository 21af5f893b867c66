"""float16 / bfloat16 decoder output without a GPU: the host rounding the
CPU emulation stores with, the decode kernels' bodies at both reduced types
(tests/emu), and the reader logic of ``open(..., dtype=...)`` on the CPU
emulation backend (tests/cpu_backend.py).  The rule throughout: a reduced
result is the float32 result converted with torch's ``.to(dtype)``, bit for
bit, NaN by position only.  The same reads run on the B200 in
tests/test_gpu_reduced.py."""
import ctypes
import io
import os
import socket
import sys

import numpy as np
import pytest
import torch

import emu_build
import reduced_cases
from reduced_cases import HALF, assert_reduced

HERE = os.path.dirname(os.path.abspath(__file__))
CODES = {torch.float16: 2, torch.bfloat16: 3}       # bb_dtype


@pytest.fixture(scope='module')
def emu():
    lib = emu_build.load()
    lib.emu_round_half.restype = None
    lib.emu_round_half.argtypes = [ctypes.c_void_p, ctypes.c_int64,
                                   ctypes.c_int32, ctypes.c_void_p]
    lib.emu_reduced_error.restype = ctypes.c_char_p
    return lib


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


# ------------------------------------------------------- host rounding
def _round(emu, values, dtype):
    x = np.ascontiguousarray(values, np.float32)
    out = np.empty(x.size, np.uint16)
    emu.emu_round_half(_ptr(x), x.size, int(dtype == torch.bfloat16),
                       _ptr(out))
    return torch.from_numpy(out.view(np.int16)).view(dtype)


def _check_round(emu, values):
    x = np.ascontiguousarray(values, np.float32).ravel()
    for dtype in HALF:
        got = _round(emu, x, dtype)
        if dtype == torch.float16:
            with np.errstate(over='ignore'):
                want = torch.from_numpy(x.astype(np.float16))
        else:
            want = torch.from_numpy(x).to(torch.bfloat16)
        assert_reduced(got, want.float(), dtype)


def _level_tables():
    from baseband_b200 import levels
    tables = [levels.offset_binary(b) for b in (1, 2, 4, 8)]
    tables += [levels.mark5b(b) for b in (1, 2)]
    tables += [levels.sign_magnitude(),
               np.arange(-8, 8, dtype=np.float32),       # GSB 4 bit
               np.arange(-128, 128, dtype=np.float32)]   # int8
    return tables


def test_round_level_tables(emu):
    """Every level a decoder stores, including all 256 affine8 values
    (offset_binary(8) is what the table-free 8-bit decode computes)."""
    for table in _level_tables():
        _check_round(emu, table)
        _check_round(emu, -table)


def test_round_edges(emu):
    f16_ulp1 = 2.0 ** -10
    specials = [
        0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan,
        1 + f16_ulp1 / 2, 1 + 3 * f16_ulp1 / 2, -(1 + f16_ulp1 / 2),
        2049.0, 2051.0, 1 + 2.0 ** -8, 1 + 3 * 2.0 ** -8,   # ties
        65504.0, 65519.99, 65520.0, -65520.0, 65536.0, 1e6, -1e6,
        2.0 ** -14, 2.0 ** -14 - 2.0 ** -30, 2.0 ** -24, 2.0 ** -25,
        3 * 2.0 ** -25, 3 * 2.0 ** -26, 2.0 ** -26, 1.5 * 2.0 ** -24,
        1e-45, -1e-45, 1.17549435e-38, 3.4028235e38, -3.4028235e38]
    bits = np.array([0x7f7f0000, 0x7f7f7fff, 0x7f7f8000, 0x7f7fffff,
                     0x7f800001, 0xff800001, 0x7fc00000, 0x00000001,
                     0x807fffff, 0x477fefff, 0x477ff000, 0x33000000,
                     0x33000001, 0x387fffff, 0x38800000], np.uint32)
    _check_round(emu, np.array(specials, np.float32))
    _check_round(emu, bits.view(np.float32))
    # around every f16 rounding boundary of [2^-26, 2^17): the tie, +-1 ulp
    e = np.arange(-26, 17)
    m = np.arange(0, 1024) / 1024.0
    grid = (np.ldexp(1 + m[None, :], e[:, None])).astype(np.float32).ravel()
    half = np.ldexp(np.float32(2.0 ** -11), e).astype(np.float32)
    ties = (grid.reshape(len(e), -1) + half[:, None]).astype(np.float32)
    ties = ties.ravel().view(np.uint32)
    _check_round(emu, np.concatenate([ties, ties + 1, ties - 1])
                 .view(np.float32))


def test_round_random_patterns(emu):
    x = np.random.default_rng(20261021).integers(
        0, 2 ** 32, 10 ** 7, dtype=np.uint64).astype(np.uint32)
    _check_round(emu, x.view(np.float32))


# ------------------------------------------------- emulated kernel bodies
def _half_buffer(n):
    """n 16-bit elements, 16-byte aligned, with sentinels either side."""
    pad = 64
    buf = np.full(n + 2 * pad + 8, 0x5a5a, np.uint16)
    sh = (-buf.ctypes.data // 2) % 8
    return buf, buf[sh + pad:sh + pad + n], sh


def _check_half_out(buf, body, sh, want32, dtype):
    pad = 64
    assert np.all(buf[:sh + pad] == 0x5a5a)
    assert np.all(buf[sh + pad + body.size:] == 0x5a5a)
    got = torch.from_numpy(body.view(np.int16)).view(dtype)
    assert_reduced(got, torch.from_numpy(
        np.ascontiguousarray(want32).ravel()), dtype)


def _bitfield_case(emu, case):
    from bitfield_cases import make_decode_case
    c = make_decode_case(case)
    lv = c['levels']
    lvp = (lv.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
           if lv is not None else None)
    n = c['nsample'] * c['nthread'] * c['nelem']
    ref = np.full(n + 8, np.float32(np.nan))
    ref = ref[(-ref.ctypes.data // 4) % 4:][:n]
    args = (_ptr(c['raw']), _ptr(c['unit_offset']), c['nset'], c['nthread'],
            c['payload_nbytes'], c['bps'], c['nelem'], int(c['complex']),
            c['codec'], lvp, c['fill'], c['sample_start'], c['nsample'])
    assert emu.bb_decode_bitfield(*args, _ptr(ref), None) == 0
    for dtype in HALF:
        buf, body, sh = _half_buffer(n)
        rc = emu.bb_decode_bitfield_typed(*args, CODES[dtype], _ptr(body),
                                          None)
        assert rc == 0, emu.emu_reduced_error()
        _check_half_out(buf, body, sh, ref, dtype)


def test_bitfield_cases(emu):
    from bitfield_cases import DECODE_CASES
    for case in DECODE_CASES:
        _bitfield_case(emu, case)


def test_bitfield_matrix(emu):
    """Every decode cell of the planner (all kernel instances, partly
    filled last rounds, invalid units, fill -0.0 / NaN) at both types."""
    from bitfield_cases import matrix_cases
    for case in matrix_cases()[0]:
        _bitfield_case(emu, case)


@pytest.mark.parametrize('case', __import__('mark4_cases').FRAME_CASES,
                         ids=lambda c: c[0])
def test_mark4_frames(emu, case):
    from mark4_cases import make_frames, oracle_frames
    from baseband_b200 import levels
    cid, mode, nframe, invalid, start, count, fill = case
    c = make_frames(mode, nframe, invalid, cid)
    want = oracle_frames(c, fill, start, count)
    lv = np.ascontiguousarray(levels.sign_magnitude(), np.float32)
    for dtype in HALF:
        buf, body, sh = _half_buffer(want.size)
        rc = emu.bb_mark4_decode_typed(
            _ptr(c['raw']), _ptr(c['unit_offset']), nframe, c['nchan'],
            c['fanout'], int(c['ft']),
            lv.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), fill, start,
            want.shape[0], CODES[dtype], _ptr(body), None)
        assert rc == 0, emu.emu_reduced_error()
        _check_half_out(buf, body, sh, want, dtype)


def _int8_cases():
    import int8_cases
    return ([('t', c) for c in int8_cases.CASES]
            + [('tf', c) for c in int8_cases.TF_CASES])


@pytest.mark.parametrize('kind,case', _int8_cases(),
                         ids=lambda c: c if isinstance(c, str) else c[0])
def test_int8(emu, kind, case):
    """Transposed (fast tile and generic) and time-first decodes; untouched
    output (invalid units) keeps its sentinel."""
    import int8_cases
    if kind == 't':
        c = int8_cases.make_case(case)
        want = int8_cases.oracle_decode(c)
    else:
        c = int8_cases.make_tf_case(case)
        want = int8_cases.oracle_tf_decode(c)
    for dtype in HALF:
        buf, body, sh = _half_buffer(want.size)
        body[:] = 0x7e00 if dtype == torch.float16 else 0x7fc0   # NaN
        if kind == 't':
            rc = emu.bb_decode_int8_transposed_typed(
                _ptr(c['raw']), _ptr(c['unit_offset']), c['nunit'],
                c['nrow'], c['ncol'], c['ib'], _ptr(c['col_begin']),
                _ptr(c['col_end']), _ptr(c['out_col0']), CODES[dtype],
                _ptr(body), None)
        else:
            rc = emu.bb_decode_int8_timefirst_typed(
                _ptr(c['raw']), _ptr(c['unit_offset']), c['nunit'],
                c['nsample'], c['nchan'], c['npol'], c['ib'],
                _ptr(c['t_begin']), _ptr(c['t_end']), _ptr(c['out_t0']),
                CODES[dtype], _ptr(body), None)
        assert rc == 0
        _check_half_out(buf, body, sh, want, dtype)


# ------------------------------------------------------------ reader logic
@pytest.fixture
def backend(monkeypatch):
    import cpu_backend
    cpu_backend.install(monkeypatch)


def test_dtype_argument(backend):
    import baseband_b200 as bb
    from conftest import sample_path
    path = sample_path('sample.vdif')
    for arg, want in ((None, np.dtype(np.float32)),
                      ('float32', np.dtype(np.float32)),
                      (torch.float32, np.dtype(np.float32)),
                      ('float16', torch.float16),
                      (torch.float16, torch.float16),
                      ('bfloat16', torch.bfloat16),
                      (torch.bfloat16, torch.bfloat16)):
        with bb.vdif.open(path, 'rs', dtype=arg) as fh:
            assert fh.dtype == want
    for bad in ('float64', 'half', torch.float64, np.float16, 16, [1]):
        with pytest.raises(ValueError):
            bb.vdif.open(path, 'rs', dtype=bad)
    # a float32 reader's results are unchanged (numpy, float32)
    with bb.vdif.open(path, 'rs', dtype='float32') as fh:
        data = fh.read(10)
        assert isinstance(data, np.ndarray) and data.dtype == np.float32


def test_writers_refuse_dtype(backend):
    import baseband_b200 as bb
    from conftest import sample_path
    G = reduced_cases.GSB
    h = bb.vdif.open(sample_path('sample.vdif'), 'rs').header0
    h5 = bb.mark5b.open(sample_path('sample.m5b'), 'rs', sample_rate=32e6,
                        kday=56000, nchan=8).header0
    h4 = bb.mark4.open(sample_path('sample.m4'), 'rs', decade=2010).header0
    hg = bb.guppi.open(sample_path('sample_puppi.raw'), 'rs').header0
    hd = bb.dada.open(sample_path('sample.dada'), 'rs').header0
    gsb = bb.gsb.open(os.path.join(G, 'sample_gsb_rawdump.timestamp'), 'rs',
                      raw=os.path.join(G, 'sample_gsb_rawdump.dat'))
    writers = [
        lambda: bb.vdif.open(io.BytesIO(), 'ws', header0=h, nthread=8,
                             sample_rate=32e6, dtype='float16'),
        lambda: bb.mark5b.open(io.BytesIO(), 'ws', header0=h5, nchan=8,
                               sample_rate=32e6, dtype='float16'),
        lambda: bb.mark4.open(io.BytesIO(), 'ws', header0=h4,
                              sample_rate=32e6, dtype='float16'),
        lambda: bb.guppi.open(io.BytesIO(), 'ws', header0=hg,
                              dtype='float16'),
        lambda: bb.dada.open(io.BytesIO(), 'ws', header0=hd,
                             dtype='bfloat16'),
        lambda: bb.gsb.open(io.StringIO(), 'ws', raw=io.BytesIO(),
                            header0=gsb.header0, sample_rate=gsb.sample_rate,
                            payload_nbytes=gsb.payload_nbytes,
                            dtype='float16'),
    ]
    for make in writers:
        with pytest.raises(TypeError):
            make()


@pytest.mark.parametrize('name', sorted(reduced_cases.STREAMS))
def test_stream_reads(backend, name):
    reduced_cases.check_stream(name, 'cpu', fills=(-0., float('nan'), 1e6))


def test_out_variants(backend):
    reduced_cases.check_out_variants('cpu', pinned=False)


def test_shapes_and_subsets(backend):
    reduced_cases.check_shapes_and_subsets('cpu')


def test_small_reads_and_pickle(backend):
    reduced_cases.check_small_reads_and_pickle()


def test_file_list_and_template(backend, tmp_path):
    """``dtype`` reaches the reader when ``open`` is given a list of files."""
    import baseband_b200 as bb
    from conftest import sample_path
    raw = np.fromfile(sample_path('sample.vdif'), np.uint8)
    names = [str(tmp_path / 'part{}.vdif'.format(i)) for i in range(2)]
    raw[:8 * 5032].tofile(names[0])
    raw[8 * 5032:].tofile(names[1])
    want = bb.vdif.open(sample_path('sample.vdif'), 'rs').read()
    with bb.vdif.open(names, 'rs', dtype='bfloat16') as fh:
        assert_reduced(fh.read(), want, torch.bfloat16)


# --------------------------------------------------------- sharded read
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, results):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port),
                      RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    from _pytest.monkeypatch import MonkeyPatch
    import cpu_backend
    patch = MonkeyPatch()
    cpu_backend.install(patch)
    import baseband_b200 as bb
    from baseband_b200 import parallel, synthetic
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        raw = synthetic.vdif_stream(7, 16, 8000, seed=21, invalid=[5, 40])
        ref = bb.vdif.open(io.BytesIO(raw.tobytes()), 'rs', sample_rate=64e6,
                           device='cpu').read()
        fh = bb.vdif.open(io.BytesIO(raw.tobytes()), 'rs', sample_rate=64e6,
                          device='cpu', dtype='float16')
        whole, span = parallel.read_sharded(fh, gather=True)
        ok = span == (0, ref.shape[0]) and whole.dtype == torch.float16
        try:
            assert_reduced(whole, ref, torch.float16)
        except AssertionError:
            ok = False
        results[rank] = bool(ok)
    finally:
        dist.destroy_process_group()
        patch.undo()


@pytest.mark.timeout(300)
def test_read_sharded_gather_float16():
    import torch.multiprocessing as mp
    world = 2
    port = _free_port()
    ctx = mp.get_context('spawn')
    with ctx.Manager() as manager:
        results = manager.dict()
        procs = [ctx.Process(target=_worker, args=(r, world, port, results))
                 for r in range(world)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(240)
        assert all(p.exitcode == 0 for p in procs), [p.exitcode
                                                     for p in procs]
        out = dict(results)
    assert all(out[r] for r in range(world))
