"""float16 / bfloat16 encoder input: every encode of a 16-bit value must give
exactly the bytes the float32 encoder gives for the value widened to float32
(``x.float()``; widening is exact).  Kernel-level cases (every 16-bit bit
pattern through every quantiser and layout, every encode cell of the
planner, input alignment), stream writers of every format and the
``read(dtype=..., on_device=writer.write)`` round trip.  Shared by
tests/test_host_reduced_encode.py (CPU emulation backend, ``dev='cpu'``) and
tests/test_gpu_reduced_encode.py (B200)."""
import io
import math
import warnings

import numpy as np
import torch

import baseband_b200 as bb
import reduced_cases
from baseband_b200 import kernels

HALF = (torch.float16, torch.bfloat16)
SENTINEL = 64 << 10                 # bytes of sentinel on each side of dst
FILL = 0x5A


def all_patterns(dtype):
    """All 65 536 values of a 16-bit type (host tensor)."""
    return torch.arange(-32768, 32768, dtype=torch.int32).to(
        torch.int16).view(dtype)


def widen(x):
    """Exact float32 value of every element of a float16 / bfloat16 tensor,
    NaN with its sign, computed on the host from the bits."""
    bits = x.detach().cpu().contiguous().view(torch.int16).numpy()
    if x.dtype == torch.bfloat16:
        f = (bits.astype(np.uint16).astype(np.uint32) << 16).view(np.float32)
    else:
        f = bits.view(np.float16).astype(np.float32)
    return torch.from_numpy(f).to(x.device)


def _dst(nbytes, dev):
    """A ``nbytes`` view of a buffer with SENTINEL bytes either side."""
    buf = torch.full((nbytes + 2 * SENTINEL,), FILL, dtype=torch.uint8,
                     device=dev)
    return buf, buf[SENTINEL:SENTINEL + nbytes]


def _aligned(values, dev, align=16):
    """``values`` on ``dev`` in a fresh buffer whose data is ``align``-byte
    aligned (torch's allocators align more; this makes it explicit)."""
    n, es = values.numel(), values.element_size()
    buf = torch.empty(n + align, dtype=values.dtype, device=dev)
    shift = (-buf.data_ptr() % align) // es
    out = buf[shift:shift + n].view(values.shape)
    out.copy_(values.to(dev))
    return out


def check_same_encode(encode, x16, dst_nbytes, dev, untouched=()):
    """``encode(data, dst)`` of ``x16`` and of its float32 widening give the
    same bytes; sentinels and the byte ranges ``untouched`` keep FILL."""
    want_buf, want = _dst(dst_nbytes, dev)
    encode(_aligned(widen(x16), dev), want)
    got_buf, got = _dst(dst_nbytes, dev)
    encode(_aligned(x16, dev), got)
    if not torch.equal(got_buf, want_buf):
        bad = (got_buf != want_buf).nonzero().reshape(-1)
        raise AssertionError('{} of {} bytes differ, first at {}'.format(
            bad.numel(), got_buf.numel(), int(bad[0]) - SENTINEL))
    assert bool((got_buf[:SENTINEL] == FILL).all())
    assert bool((got_buf[SENTINEL + dst_nbytes:] == FILL).all())
    for a, b in untouched:
        assert bool((got[a:b] == FILL).all()), (a, b)


def _tile(x, n):
    reps = -(-n // x.numel())
    return x.repeat(reps)[:n]


# ------------------------------------------------- exhaustive bit patterns
# bit-field shapes (nthread, nelem): RUN / RUNQ, ROWGROUP4, ROWWORD4,
# ROWWORD2 / ROWGROUP2, SCALAR
BITFIELD_SHAPES = ((1, 1), (16, 1), (4, 1), (2, 2), (3, 1))
QUANTISERS = [(kernels.QUANT_OFFSET_BINARY, b) for b in (1, 2, 4, 8)] + [
    (kernels.QUANT_MARK5B, 1), (kernels.QUANT_MARK5B, 2),
    (kernels.QUANT_SINT, 4), (kernels.QUANT_SINT, 8)]


def exhaustive_bitfield(dev, dtype, report=None):
    x = all_patterns(dtype)
    for nthread, nelem in BITFIELD_SHAPES:
        rowlen = nthread * nelem
        for quant, bps in QUANTISERS:
            nset = 2
            m = 32 // math.gcd(32, nelem * bps)     # whole 32-bit words
            spf = -(-x.numel() // (nset * rowlen * m)) * m
            payload = spf * nelem * bps // 8
            data = _tile(x, nset * spf * rowlen)
            stride = payload + 32
            uo = torch.arange(nset * nthread, dtype=torch.int64) * stride + 32
            uo[1] = -1                              # an invalid unit
            uo = uo.to(dev)

            def encode(d, dst):
                kernels.encode_bitfield(d, dst, uo, nset, nthread, payload,
                                        bps, nelem, quant)
            check_same_encode(encode, data, nset * nthread * stride + 32,
                              dev, untouched=[(32 + stride, 32 + 2 * stride)])
            if report is not None and nthread == 1:
                # numpy float16 goes through float64: count the output bytes
                # its float64 encode changes (documentation, not a rule)
                _, a = _dst(nset * stride + 32, dev)
                _, b = _dst(nset * stride + 32, dev)
                w = widen(data)
                encode(_aligned(w, dev), a)
                encode(_aligned(w.double(), dev), b)
                report[(dtype, quant, bps)] = int((a != b).sum())


def exhaustive_mark4(dev, dtype):
    from mark4_cases import MODES
    x = all_patterns(dtype)
    for mode, (nchan, fanout, ft) in MODES.items():
        wb = nchan * 2 * fanout // 8
        nframe = 1
        spf = 20000 * fanout
        data = _tile(x, nframe * spf * nchan)
        uo = torch.tensor([160 * wb], dtype=torch.int64, device=dev)

        def encode(d, dst):
            kernels.mark4_encode(d, dst, uo, nframe, nchan, fanout, ft)
        check_same_encode(encode, data, 20000 * wb, dev,
                          untouched=[(0, 160 * wb)])


# int8 transposed (nunit, nrow, ncol, ib): fast tiles with interior and edge
# tiles (complex and real), and odd nrow (the plain tile kernel)
INT8_T_SHAPES = ((2, 128, 300, 2), (1, 130, 520, 1), (1, 67, 300, 2))
# time-first (nunit, nsample, nchan, npol, ib): vector path at npol 1 / 2 /
# 4, and the one-value-per-item path
INT8_TF_SHAPES = ((2, 1024, 16, 2, 2), (1, 512, 32, 4, 2), (1, 2048, 32, 1, 1),
                  (2, 700, 3, 2, 2), (1, 1000, 5, 3, 1))


def exhaustive_int8(dev, dtype):
    x = all_patterns(dtype)
    for nunit, nrow, ncol, ib in INT8_T_SHAPES:
        unit = nrow * ncol * ib
        data = _tile(x, nunit * unit)
        uo = torch.arange(nunit, dtype=torch.int64) * (unit + 64) + 8
        uo = uo.to(dev)

        def encode(d, dst):
            kernels.encode_int8_transposed(d, dst, uo, nunit, nrow, ncol, ib)
        check_same_encode(encode, data, nunit * (unit + 64) + 8, dev)
    for nunit, nsample, nchan, npol, ib in INT8_TF_SHAPES:
        unit = nsample * nchan * npol * ib
        data = _tile(x, nunit * unit)
        uo = torch.arange(nunit, dtype=torch.int64) * (unit + 64) + 16
        uo = uo.to(dev)

        def encode(d, dst):
            kernels.encode_int8_timefirst(d, dst, uo, nunit, nsample, nchan,
                                          npol, ib)
        check_same_encode(encode, data, nunit * (unit + 64) + 16, dev)


# ------------------------------------------------------ every encode cell
def matrix_cell(dev, case):
    """One float32-keyed encode cell of ``bitfield_cases.matrix_cases()``,
    its data rounded to each 16-bit type."""
    from bitfield_cases import make_encode_case
    c = make_encode_case(case)
    uo = torch.from_numpy(c['unit_offset']).to(dev)
    untouched = [(int(t), int(t) + c['payload_nbytes'])
                 for t, u in zip(c['truth'], c['unit_offset']) if u < 0]

    def encode(d, dst):
        kernels.encode_bitfield(d, dst, uo, c['nset'], c['nthread'],
                                c['payload_nbytes'], c['bps'], c['nelem'],
                                c['quantiser'])
    x32 = torch.from_numpy(np.ascontiguousarray(c['data']))
    for dtype in HALF:
        check_same_encode(encode, x32.to(dtype), c['dst_nbytes'], dev,
                          untouched)


# ------------------------------------------------------------- alignment
def check_alignment(dev):
    """16-bit input must be 8-byte aligned: a 4-byte aligned pointer is
    refused with ValueError, an 8-byte aligned view encodes correctly."""
    import pytest
    nthread, payload, bps = 16, 800, 2
    spf = payload * 8 // bps
    uo = (torch.arange(nthread, dtype=torch.int64) * (payload + 32)
          + 32).to(dev)
    for dtype in HALF:
        base = _aligned(torch.randn(spf * nthread + 8).to(dtype), dev)
        dst = torch.zeros(nthread * (payload + 32) + 32, dtype=torch.uint8,
                          device=dev)
        with pytest.raises(ValueError):
            kernels.encode_bitfield(base[2:2 + spf * nthread], dst, uo, 1,
                                    nthread, payload, bps, 1)
        with pytest.raises(ValueError):
            kernels.mark4_encode(base[2:], dst, uo[:1], 1, 8, 4)

        def encode(d, dst):
            kernels.encode_bitfield(d, dst, uo, 1, nthread, payload, bps, 1)
        view = base[4:4 + spf * nthread]
        want_buf, want = _dst(dst.numel(), dev)
        encode(_aligned(widen(view), dev), want)
        got_buf, got = _dst(dst.numel(), dev)
        encode(view, got)
        assert torch.equal(got_buf, want_buf)


# ---------------------------------------------------------------- writers
class _Sink(io.BytesIO):
    """A file whose bytes can be read after the writer closed it."""
    def close(self):
        pass


def _writer(name, fh, dev):
    """A writer of the same stream as reader ``fh``: (writer, bytes())."""
    h0 = fh.header0
    if name == 'gsb_phased':
        bufs = [[_Sink(), _Sink()], [_Sink(), _Sink()]]
        fw = bb.gsb.open(io.StringIO(), 'ws', raw=bufs, header0=h0,
                         sample_rate=fh.sample_rate, payload_nbytes=8192,
                         device=dev)
        return fw, lambda: b''.join(b.getvalue() for g in bufs for b in g)
    buf = _Sink()
    if name.startswith('vdif'):
        fw = bb.vdif.open(buf, 'ws', header0=h0, nthread=fh.sample_shape[0],
                          sample_rate=fh.sample_rate, device=dev)
    elif name.startswith('mark5b'):
        fw = bb.mark5b.open(buf, 'ws', header0=h0, nchan=fh.sample_shape[0],
                            sample_rate=fh.sample_rate, device=dev)
    elif name.startswith('mark4'):
        fw = bb.mark4.open(buf, 'ws', header0=h0, sample_rate=fh.sample_rate,
                           device=dev)
    elif name.startswith('guppi'):
        fw = bb.guppi.open(buf, 'ws', header0=h0, device=dev)
    elif name.startswith('dada'):
        if h0.get('INSTRUMENT') == 'MKBF':
            # the sample's header describes a much longer file: one frame of
            # the heaps it has
            h0 = h0.copy()
            h0.mutable = True
            h0.payload_nbytes = fh.shape[0] * h0['NPOL'] * h0['NCHAN'] * 2
        fw = bb.dada.open(buf, 'ws', header0=h0, device=dev)
    else:
        fw = bb.gsb.open(io.StringIO(), 'ws', raw=buf, header0=h0,
                         sample_rate=fh.sample_rate, payload_nbytes=4096,
                         device=dev)
    return fw, buf.getvalue


def _guppi_synth():
    """GUPPI without overlap (a writer needs none)."""
    from baseband_b200 import synthetic
    raw, _ = synthetic.guppi_stream(5, nchan=8, npol=2, samples_per_frame=64,
                                    overlap=0)
    data = raw.tobytes()
    return lambda **kw: bb.guppi.open(io.BytesIO(data), 'rs', **kw)


def _opener(name):
    if name == 'guppi_synth':
        return _guppi_synth()
    return reduced_cases.STREAMS[name][0]()


WRITER_STREAMS = ('vdif_sample_invalid', 'vdif_complex', 'mark5b_invalid',
                  'mark4_sample', 'guppi_synth', 'dada_sample', 'dada_mkbf',
                  'gsb_rawdump', 'gsb_phased')


def to_half(x32, dtype):
    """float32 / complex64 samples -> the 16-bit form a ``dtype`` reader
    returns (complex32, or bfloat16 with a trailing (re, im) axis)."""
    if not x32.is_complex():
        return x32.to(dtype)
    pairs = torch.view_as_real(x32).to(dtype)
    return torch.view_as_complex(pairs) if dtype == torch.float16 else pairs


def as_float(x16, complex_data):
    """The float32 / complex64 widening of a 16-bit writer input."""
    if x16.dtype == torch.complex32:
        x16 = torch.view_as_real(x16)
    w = widen(x16)
    return torch.view_as_complex(w.contiguous()) if complex_data else w


def _write(name, fh, dev, pieces):
    fw, get = _writer(name, fh, dev)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')          # closing a partial frame
        for piece, valid in pieces:
            fw.write(piece, valid=valid)
        fw.close()
    return get()


def check_writer(name, dev):
    """Writing the 16-bit forms of a stream gives the file that writing
    their float32 widening does: whole, in mixed-type pieces, with a
    partial last frame, from a misaligned view, with valid=False, from the
    host."""
    opener = _opener(name)
    with opener() as fh:
        x32 = torch.from_numpy(np.ascontiguousarray(fh.read()))
        cplx = fh.complex_data
        spf = fh.samples_per_frame
        n = x32.shape[0]
        k = min(spf + spf // 2 + 1, n // 2)     # a piece boundary mid-frame
        for dtype in HALF:
            x16 = to_half(x32, dtype).to(dev)
            w = as_float(x16, cplx).to(dev)
            part = max(1, n - spf // 2 - 1)       # leaves a partial frame
            lay = torch.empty((n + 1,) + tuple(x16.shape[1:]),
                              dtype=x16.dtype, device=dev)
            lay[1:] = x16
            runs = [
                ([(x16[:k], True), (x16[k:], True)],
                 [(w[:k], True), (w[k:], True)]),
                ([(x16[:k], True), (w[k:], True)],            # mixed types
                 [(w[:k], True), (w[k:], True)]),
                ([(x16[:part], True)], [(w[:part], True)]),
                ([(lay[1:], True)], [(w, True)]),             # misaligned
                ([(x16[:k], True), (x16[k:], False)],
                 [(w[:k], True), (w[k:], False)]),
                ([(x16.cpu(), True)], [(w.cpu(), True)]),     # host input
            ]
            if x16.dtype == torch.bfloat16 or not cplx:
                # float16 with bfloat16 promotes to float32
                other = (x32[k:].to(torch.float16) if not cplx else
                         torch.view_as_complex(torch.view_as_real(
                             x32[k:]).to(torch.float16)))
                runs.append(([(x16[:k], True), (other.to(dev), True)],
                             [(w[:k], True),
                              (as_float(other, cplx).to(dev), True)]))
            for got_pieces, want_pieces in runs:
                got = _write(name, fh, dev, got_pieces)
                want = _write(name, fh, dev, want_pieces)
                assert got == want, (name, dtype)


def check_type_errors(dev):
    """Real and complex streams refuse the other kind of 16-bit input."""
    import pytest
    real = reduced_cases.STREAMS['vdif_sample_invalid'][0]()
    cplx = reduced_cases.STREAMS['vdif_complex'][0]()
    with real() as fh:
        x = torch.from_numpy(fh.read())
        fw, _ = _writer('vdif_sample_invalid', fh, dev)
        with pytest.raises(ValueError):
            fw.write(torch.view_as_complex(
                torch.stack([x, x], -1).to(torch.float16)))
    with cplx() as fh:
        x = torch.from_numpy(fh.read())
        fw, _ = _writer('vdif_complex', fh, dev)
        for bad in (x.real.to(torch.float16), x.real.to(torch.bfloat16),
                    torch.view_as_real(x)[..., :1].to(torch.bfloat16)):
            with pytest.raises(ValueError):
                fw.write(bad.to(dev))


# ------------------------------------------------------------- round trip
ROUND_TRIP_STREAMS = WRITER_STREAMS


def check_round_trip(name, dev):
    """``read(dtype=d, on_device=writer.write)`` writes what the float32
    round trip writes, at both 16-bit types."""
    opener = _opener(name)
    outs = {}
    for dtype in (None,) + HALF:
        with opener(device=dev, dtype=dtype) as fh:
            fw, get = _writer(name, fh, dev)
            fh.read(on_device=fw.write)
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                fw.close()
            outs[dtype] = get()
    for dtype in HALF:
        assert outs[dtype] == outs[None], (name, dtype)
