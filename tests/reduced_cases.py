"""Reduced-precision stream reads (``open(..., dtype='float16' /
'bfloat16')``): every read must equal the same float32 read converted
elementwise with torch's ``.to(dtype)``, bit for bit, -0.0 and +-inf
included; NaN only by position.  Shared by tests/test_host_reduced.py (CPU
emulation backend, ``dev='cpu'``) and tests/test_gpu_reduced.py (B200)."""
import io
import os
import pickle
import warnings

import numpy as np
import torch

import baseband_b200 as bb
from baseband_b200 import synthetic
from conftest import sample_path

HALF = (torch.float16, torch.bfloat16)
FILLS = (0., -999., -0., float('nan'), 1e6)
GSB = os.path.join(os.path.dirname(sample_path('x')), 'gsb')


def as_pairs(t, device='cpu'):
    """float32 / complex64 / half result -> tensor of real elements on
    ``device`` (complex as a trailing (re, im) axis)."""
    t = torch.from_numpy(np.ascontiguousarray(t)) if isinstance(
        t, np.ndarray) else t
    t = t.to(device)
    return torch.view_as_real(t) if t.is_complex() else t


def assert_reduced(got, want32, dtype):
    """``got`` is ``want32.to(dtype)`` under the exactness rule (compared
    where ``got`` lives)."""
    dev = got.device if isinstance(got, torch.Tensor) else 'cpu'
    g = as_pairs(got, dev)
    exp = as_pairs(want32, dev).to(dtype)
    assert g.dtype == dtype, (g.dtype, dtype)
    assert tuple(g.shape) == tuple(exp.shape), (g.shape, exp.shape)
    gn, en = torch.isnan(g.float()), torch.isnan(exp.float())
    assert torch.equal(gn, en), 'NaN positions differ'
    gb, eb = g.view(torch.int16)[~gn], exp.view(torch.int16)[~en]
    if not torch.equal(gb, eb):
        bad = (gb != eb).nonzero()[:5].reshape(-1)
        raise AssertionError('{} of {} values differ, e.g. at {}: {} vs {}'
                             .format(int((gb != eb).sum()), gb.numel(),
                                     bad.tolist(), gb[bad].tolist(),
                                     eb[bad].tolist()))


def result_type(dtype, complex_data):
    if not complex_data:
        return dtype
    return torch.complex32 if dtype == torch.float16 else torch.bfloat16


# --------------------------------------------------------------- streams
# name -> (opener(**kw), takes fill_value, reads(n) -> [(start, count)])
def _vdif_sample_invalid():
    raw = np.fromfile(sample_path('sample.vdif'), np.uint8).copy()
    frames = raw.reshape(16, 5032)
    tid = (frames[:, 12:16].view('<u4')[:, 0] >> 16) & 0x3ff
    for i in range(8):
        if tid[i] in (1, 4, 7):
            frames[i, 3] |= 0x80
    data = raw.tobytes()
    return lambda **kw: bb.vdif.open(io.BytesIO(data), 'rs',
                                     chunk_nbytes=8 * 5032, **kw)


def _vdif_synth16():
    raw = synthetic.vdif_stream(23, 16, 8000, seed=5, invalid=[3, 77, 78])
    data = raw.tobytes()
    return lambda **kw: bb.vdif.open(io.BytesIO(data), 'rs', sample_rate=64e6,
                                     chunk_nbytes=16 * 8032 * 3, **kw)


def _vdif_complex():
    return lambda **kw: bb.vdif.open(sample_path('sample_arochime.vdif'),
                                     'rs', sample_rate=1e6, **kw)


def _vdif_irregular():
    """Dropped and duplicated frames: read through the GPU frame index."""
    nset, nthread = 9, 8
    raw = synthetic.vdif_stream(nset, nthread, 5000, seed=41,
                                thread_order=np.arange(nthread))
    frames = raw.reshape(nset * nthread, 5032)
    keep = [i for i in range(nset * nthread) if i not in (3, 20, 21, 22, 47)]
    lossy = frames[keep]
    data = np.concatenate([lossy[:30], lossy[29:30], lossy[30:]]).tobytes()

    def opener(**kw):
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            return bb.vdif.open(io.BytesIO(data), 'rs', sample_rate=32e6,
                                chunk_nbytes=2 * nthread * 5032, **kw)
    return opener


def _mark5b_invalid():
    raw, _ = synthetic.mark5b_stream(40, invalid_fraction=0.2, seed=77)
    data = raw.tobytes()
    return lambda **kw: bb.mark5b.open(io.BytesIO(data), 'rs', nchan=16,
                                       sample_rate=16e6, kday=56000,
                                       chunk_nbytes=7 * 10016, **kw)


def _mark4_sample():
    return lambda **kw: bb.mark4.open(sample_path('sample.m4'), 'rs',
                                      decade=2010, **kw)


def _guppi_sample():
    return lambda **kw: bb.guppi.open(sample_path('sample_puppi.raw'), 'rs',
                                      **kw)


def _guppi_overlap():
    raw, _ = synthetic.guppi_stream(5, nchan=8, npol=2, samples_per_frame=64,
                                    overlap=8)
    data = raw.tobytes()
    return lambda **kw: bb.guppi.open(io.BytesIO(data), 'rs', **kw)


def _dada_sample():
    return lambda **kw: bb.dada.open(sample_path('sample.dada'), 'rs',
                                     chunk_nbytes=3000, **kw)


def _dada_mkbf():
    return lambda **kw: bb.dada.open(sample_path('sample_mkbf.dada'), 'rs',
                                     squeeze=False, **kw)


def _gsb_rawdump():
    return lambda **kw: bb.gsb.open(
        os.path.join(GSB, 'sample_gsb_rawdump.timestamp'), 'rs',
        raw=os.path.join(GSB, 'sample_gsb_rawdump.dat'),
        sample_rate=1e8 / 3 / 2 ** 10, payload_nbytes=4096,
        chunk_nbytes=3 * 4096, **kw)


def _gsb_phased():
    raw = [[os.path.join(GSB, 'sample_gsb_phased.Pol-%s%d.dat' % (p, k))
            for k in (1, 2)] for p in 'LR']
    return lambda **kw: bb.gsb.open(
        os.path.join(GSB, 'sample_gsb_phased.timestamp'), 'rs', raw=raw,
        sample_rate=1e8 / 3 / 2 ** 19, payload_nbytes=8192,
        chunk_nbytes=2 * 4 * 8192, **kw)


def _partial(n):
    """Whole stream, a read starting and ending inside frames, a tail."""
    mid = min(n // 3 + 1, n - 1)
    return [(0, n), (mid, min(n // 3 + 5, n - mid)), (max(0, n - 7), min(7, n))]


STREAMS = {
    'vdif_sample_invalid': (_vdif_sample_invalid, True, _partial),
    'vdif_synth16': (_vdif_synth16, True, _partial),
    'vdif_complex': (_vdif_complex, True, _partial),
    'vdif_irregular': (_vdif_irregular, True, _partial),
    'mark5b_invalid': (_mark5b_invalid, True, _partial),
    'mark4_sample': (_mark4_sample, True, _partial),
    'guppi_sample': (_guppi_sample, False, _partial),
    'guppi_overlap': (_guppi_overlap, False, _partial),
    'dada_sample': (_dada_sample, False, _partial),
    'dada_mkbf': (_dada_mkbf, False, _partial),
    'gsb_rawdump': (_gsb_rawdump, False, _partial),
    'gsb_phased': (_gsb_phased, False, _partial),
}


def check_stream(name, dev, dtypes=HALF, fills=FILLS):
    """Every read of stream ``name`` at ``dtypes``, with device output
    (``dev``) and host output, against the float32 read."""
    make, has_fill, reads = STREAMS[name]
    opener = make()
    for fill in (fills if has_fill else (None,)):
        kw = {} if fill is None else {'fill_value': fill}
        for device in (dev, None):
            with opener(device=device, **kw) as ref:
                spans = reads(ref.shape[0])
                want = []
                for start, count in spans:
                    ref.seek(start)
                    want.append(ref.read(count))
            for dtype in dtypes:
                with opener(device=device, dtype=dtype, **kw) as fh:
                    assert fh.dtype == result_type(dtype, fh.complex_data)
                    for (start, count), w in zip(spans, want):
                        fh.seek(start)
                        got = fh.read(count)
                        assert isinstance(got, torch.Tensor)
                        assert fh.tell() == start + count
                        assert_reduced(got, w, dtype)


def check_out_variants(dev, pinned):
    """read(out=...): a device tensor, a (pinned) host tensor, a pageable
    numpy float16 array (staged copy), and a float32 reader handed a half
    tensor, which decodes straight into it."""
    opener = _vdif_synth16()
    with opener(fill_value=2.5) as ref:
        ref.seek(1001)
        want = ref.read(70001)
    for dtype in HALF:
        with opener(fill_value=2.5, device=dev, dtype=dtype) as fh:
            fh.seek(1001)
            out = torch.empty(want.shape, dtype=dtype, device=dev)
            assert fh.read(out=out) is out
            assert_reduced(out, want, dtype)
        with opener(fill_value=2.5, dtype=dtype) as fh:
            fh.seek(1001)
            out = torch.empty(want.shape, dtype=dtype)
            if pinned:
                out = out.pin_memory()
            assert fh.read(out=out) is out
            assert_reduced(out, want, dtype)
        # the old path (decode to float32, then torch converts) and the
        # native one give the same values
        for device in (dev, None):
            with opener(fill_value=2.5, device=device) as fh:
                fh.seek(1001)
                out = torch.empty(want.shape, dtype=dtype,
                                  device=device or 'cpu')
                if pinned and device is None:
                    out = out.pin_memory()
                assert fh.read(out=out) is out
                assert_reduced(out, want, dtype)
    with opener(fill_value=2.5, dtype='float16') as fh:
        fh.seek(1001)
        out = np.empty(want.shape, np.float16)       # 2.2 MB: staged
        assert fh.read(out=out) is out
        assert_reduced(out, want, torch.float16)
        with np.testing.assert_raises(TypeError):
            fh.read(out=np.empty((5, 16), np.float32))
    # complex: complex32 and the bfloat16 (re, im) axis
    copen = _vdif_complex()
    with copen() as ref:
        want = ref.read()
    with copen(device=dev, dtype='float16') as fh:
        out = torch.empty(want.shape, dtype=torch.complex32, device=dev)
        assert fh.read(out=out) is out
        assert_reduced(out, want, torch.float16)
    with copen(device=dev) as fh:                  # float32 reader, native
        out = torch.empty(want.shape, dtype=torch.complex32, device=dev)
        assert fh.read(out=out) is out
        assert_reduced(out, want, torch.float16)
    with copen(device=dev, dtype='bfloat16') as fh:
        out = torch.empty(tuple(want.shape) + (2,), dtype=torch.bfloat16,
                          device=dev)
        assert fh.read(out=out) is out
        assert_reduced(out, want, torch.bfloat16)


def check_shapes_and_subsets(dev):
    """Result types and shapes, squeeze / subset, the on_device hook."""
    want = bb.vdif.open(sample_path('sample.vdif'), 'rs').read()
    for dtype, name in ((torch.float16, 'float16'),
                        (torch.bfloat16, 'bfloat16')):
        for kw, pick in (({}, want), ({'squeeze': False}, want[:, :, None]),
                         ({'subset': [1, 6]}, want[:, [1, 6]]),
                         ({'subset': 3}, want[:, 3])):
            with bb.vdif.open(sample_path('sample.vdif'), 'rs', dtype=name,
                              device=dev, **kw) as fh:
                assert fh.dtype == dtype
                assert fh.shape == pick.shape
                fh.seek(10)
                seen = []
                got = fh.read(30000, on_device=lambda p: seen.append(p.dtype))
                assert set(seen) == {dtype}
                assert_reduced(got, pick[10:30010], dtype)
    with bb.vdif.open(sample_path('sample_arochime.vdif'), 'rs',
                      sample_rate=1e6) as ref:
        cwant = ref.read()
        shape = ref.shape
    for dtype, rtype, tail in ((torch.float16, torch.complex32, ()),
                               (torch.bfloat16, torch.bfloat16, (2,))):
        with bb.vdif.open(sample_path('sample_arochime.vdif'), 'rs',
                          sample_rate=1e6, dtype=dtype, device=dev) as fh:
            assert fh.dtype == rtype and fh.shape == shape
            got = fh.read()
            assert got.dtype == rtype
            assert tuple(got.shape) == tuple(cwant.shape) + tail
            assert_reduced(got, cwant, dtype)


def check_small_reads_and_pickle():
    """Small host reads (window cache) and pickled readers keep the type."""
    want = bb.vdif.open(sample_path('sample.vdif'), 'rs').read()
    for dtype in HALF:
        with bb.vdif.open(sample_path('sample.vdif'), 'rs',
                          dtype=dtype) as fh:
            fh.seek(6)
            got = fh.read(3)
            assert isinstance(got, torch.Tensor) and got.dtype == dtype
            assert_reduced(got, want[6:9], dtype)
            fh.seek(19990)
            assert_reduced(fh.read(20), want[19990:20010], dtype)
            clone = pickle.loads(pickle.dumps(fh))
            assert clone.dtype == dtype and clone.tell() == 20010
            assert_reduced(clone.read(19990), want[20010:], dtype)
            clone.close()
    with bb.vdif.open(sample_path('sample.vdif'), 'rs',
                      dtype='float16') as fh:
        out = np.empty((40, 8), np.float16)
        fh.seek(100)
        assert fh.read(out=out) is out
        assert_reduced(out, want[100:140], torch.float16)
