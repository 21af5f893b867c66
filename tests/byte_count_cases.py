"""8-bit state counts (bb_byte_counts, tasks.state_counts on 8-bit
streams): a numpy restatement of the kernel and stream-level cases.  The
cases run on the CPU emulation backend (tests/test_host_byte_counts.py, with
the restatement standing in for the kernel) and on the GPU
(tests/test_gpu_byte_counts.py)."""
import io
import os

import numpy as np
import pytest
import torch

import baseband_b200 as bb
import cpu_backend
from baseband_b200 import synthetic
from conftest import GOLDEN, sample_path
from oracle import stream as ostream

OUT = np.load(os.path.join(GOLDEN, 'sample_outputs.npz'))
GSB = os.path.join(GOLDEN, 'samples', 'gsb')


def byte_counts(src, unit_offset, nset, nthread, payload_nbytes, nelem,
                counts, set_origin=0, sets_per_bin=None):
    """numpy restatement of bb_byte_counts (csrc/bb_counts.cu): a bincount
    of the stored bytes per unit and element."""
    buf = src.numpy()
    uo = unit_offset.numpy().reshape(nset, nthread)
    if sets_per_bin is None:
        sets_per_bin = max(1, set_origin + nset)
    if tuple(counts.shape[1:]) != (nthread, nelem, 256):
        raise ValueError('counts must have shape (nbin, nthread, nelem, 256)')
    out = counts.numpy()
    for s in range(nset):
        b = (set_origin + s) // sets_per_bin
        for t in range(nthread):
            if uo[s, t] < 0:
                continue
            x = buf[uo[s, t]:uo[s, t] + payload_nbytes].reshape(-1, nelem)
            idx = np.arange(nelem, dtype=np.int64) * 256 + x
            out[b, t] += np.bincount(idx.reshape(-1), minlength=nelem * 256
                                     ).reshape(nelem, 256)
    return counts


def install(monkeypatch):
    from baseband_b200 import kernels
    cpu_backend.install(monkeypatch)
    monkeypatch.setattr(kernels, 'byte_counts', byte_counts)


def _codes(decoded, lv):
    """Decoded samples -> the byte code behind each (through the level
    table, which is one to one)."""
    order = np.argsort(lv)
    idx = np.searchsorted(lv[order], decoded)
    idx = np.clip(idx, 0, len(lv) - 1)
    assert np.all(lv[order][idx] == decoded)
    return order[idx]


def _bincount_rows(codes, rows_per_bin):
    """codes (nsample, ...) -> (nbin, ..., 256)."""
    nbin = -(-codes.shape[0] // rows_per_bin)
    out = np.zeros((nbin,) + codes.shape[1:] + (256,), np.int64)
    flat = codes.reshape(codes.shape[0], -1)
    o = out.reshape(nbin, -1, 256)
    for b in range(nbin):
        blk = flat[b * rows_per_bin:(b + 1) * rows_per_bin]
        for k in range(flat.shape[1]):
            o[b, k] = np.bincount(blk[:, k], minlength=256)
    return out


# ------------------------------------------------------------------ VDIF
def vdif_mwa_sample():
    """The reference's 8-bit complex MWA sample: counts == the bincount of
    the codes behind its decoded golden data."""
    from baseband_b200 import tasks
    want_data = OUT['sample_mwa_vdif_data']           # (1280, 1, 2) complex
    with bb.vdif.open(sample_path('sample_mwa.vdif'), 'rs',
                      sample_rate=1.28e6) as fh:
        lv = tasks.state_levels(fh)
        assert lv.shape == (256,)
        spf = fh.samples_per_frame
        got = tasks.state_counts(fh, 4 * spf)
        assert fh.tell() == fh.shape[0]
    parts = np.stack([want_data.real, want_data.imag], -1)   # (n, 1, 2, 2)
    codes = _codes(parts.astype(np.float32), lv)
    want = _bincount_rows(codes, 4 * spf)[:, 0]       # squeezed thread axis
    assert got.shape == want.shape == (3, 2, 2, 256), got.shape
    assert np.array_equal(got, want)


def vdif_synthetic_8bit():
    """Synthetic 8-bit VDIF: several threads, complex, several channels,
    invalid frames, a thread subset, bins across chunks; and the power."""
    from baseband_b200 import tasks
    for nthread, nchan, cplx, payload in ((4, 2, True, 1024),
                                          (3, 4, False, 512),
                                          (2, 1, False, 2048)):
        nset = 7
        raw = synthetic.vdif_stream(nset, nthread, payload, bps=8,
                                    nchan=nchan, complex_data=cplx,
                                    seed=200 + nchan, invalid=[2, 9])
        frame = payload + 32
        with bb.vdif.open(io.BytesIO(raw.tobytes()), 'rs', sample_rate=1e6,
                          squeeze=False, fill_value=np.nan,
                          chunk_nbytes=3 * nthread * frame) as fh:
            lv = tasks.state_levels(fh)
            decoded = fh.read()
            spf = fh.samples_per_frame
            fh.seek(0)
            got = tasks.state_counts(fh, 2 * spf)
            fh.seek(spf)
            part = tasks.state_counts(fh, 3 * spf, count=5 * spf)
            fh.seek(0)
            power = tasks.integrated_power(fh, 2 * spf)
        if cplx:
            decoded = np.stack([decoded.real, np.where(
                np.isnan(decoded.real), np.nan, decoded.imag)], -1)
        valid = ~np.isnan(decoded)
        codes = _codes(np.where(valid, decoded, lv[0]), lv)

        def want_of(c, ok, rows):
            w = _bincount_rows(c, rows)
            # invalid samples were counted as code 0 above: take them out
            n_bad = _bincount_rows(np.where(ok, 1, 0), rows)[..., 0]
            w[..., 0] -= n_bad
            return w

        want = want_of(codes, valid, 2 * spf)
        assert got.shape == want.shape, (got.shape, want.shape)
        assert np.array_equal(got, want), (nthread, nchan, cplx)
        assert np.array_equal(part, want_of(codes[spf:6 * spf],
                                            valid[spf:6 * spf], 3 * spf))
        x = np.where(valid, decoded, np.nan).astype(np.float64) ** 2
        if cplx:
            x = x.sum(-1)
        ref = np.stack([np.nanmean(x[b * 2 * spf:(b + 1) * 2 * spf], 0)
                        for b in range(4)])
        assert np.allclose(power, ref, rtol=1e-10, atol=0)
        # a thread subset
        with bb.vdif.open(io.BytesIO(raw.tobytes()), 'rs', sample_rate=1e6,
                          squeeze=False, subset=[nthread - 1, 0]) as fh:
            sub = tasks.state_counts(fh, 2 * spf)
        assert np.array_equal(sub, want[:, [nthread - 1, 0]])


# ------------------------------------------------ two's complement, files
def _check_against_moments(fh_open, **kwargs):
    """counts and moments on the same reader agree exactly: n, the sum of
    the int8 values and of their squares."""
    from baseband_b200 import tasks
    with fh_open() as fh:
        lv = tasks.state_levels(fh)
        assert np.array_equal(lv, np.r_[0:128, -128:0].astype(np.float32))
        start = fh.tell()
        counts = tasks.state_counts(fh, **kwargs)
        end = fh.tell()
        fh.seek(start)
        n, total, sq = tasks.moments(fh, **kwargs)
        assert fh.tell() == end
        fh.seek(start)
        power = tasks.integrated_power(fh, **kwargs)
    assert counts.dtype == np.int64
    assert counts.shape == n.shape + (256,), (counts.shape, n.shape)
    lv64 = lv.astype(np.int64)
    assert np.array_equal(counts.sum(-1), n)
    assert np.array_equal((counts * lv64).sum(-1), total)
    assert np.array_equal((counts * lv64 ** 2).sum(-1), sq)
    return counts, power


def guppi_files():
    """sample_puppi.raw channels first (its overlap left out by default),
    and the same frames read time first."""
    _check_against_moments(
        lambda: bb.guppi.open(sample_path('sample_puppi.raw'), 'rs'),
        samples_per_bin=2 * 960)
    _check_against_moments(
        lambda: bb.guppi.open(sample_path('sample_puppi.raw'), 'rs',
                              squeeze=False))
    raw = open(sample_path('sample_puppi.raw'), 'rb').read()
    tf = raw.replace(b"PKTFMT  = '1SFA    '", b"PKTFMT  = 'SIMPLE  '")
    assert tf != raw
    with bb.guppi.open(io.BytesIO(tf), 'rs') as fh:
        assert not fh.header0.channels_first
    counts, _ = _check_against_moments(
        lambda: bb.guppi.open(io.BytesIO(tf), 'rs', squeeze=False))
    # the same bytes, only grouped into elements differently
    with bb.guppi.open(io.BytesIO(tf), 'rs') as fh:
        assert counts.sum() == fh._nframe * fh.samples_per_frame * 2 * 4 * 2


def guppi_synthetic():
    """Synthetic channels-first GUPPI with bins that cut the chunks."""
    from baseband_b200 import tasks
    raw, _ = synthetic.guppi_stream(5, nchan=8, npol=2, samples_per_frame=64,
                                    overlap=8)
    decoded = ostream.guppi_read(raw)                 # (nsample, npol, nchan)
    with bb.guppi.open(io.BytesIO(raw.tobytes()), 'rs', squeeze=False) as fh:
        spf = fh.samples_per_frame
        fh._chunk_nbytes = 2 * fh._frame_nbytes
        got = tasks.state_counts(fh, 3 * spf)
    body = decoded[:5 * spf]
    parts = np.stack([body.real, body.imag], -1).astype(np.int64)
    want = _bincount_rows((parts & 0xff).astype(np.int64), 3 * spf)
    assert got.shape == want.shape == (2, 2, 8, 2, 256)
    assert np.array_equal(got, want)


def dada_files():
    for name in ('sample.dada', 'sample_meerkat.dada'):
        for chunk in (None, 4096):
            _check_against_moments(
                lambda: bb.dada.open(sample_path(name), 'rs', squeeze=False,
                                     chunk_nbytes=chunk))
        _check_against_moments(lambda: bb.dada.open(sample_path(name), 'rs'))


def gsb_phased():
    raw = [[os.path.join(GSB, 'sample_gsb_phased.Pol-%s%d.dat' % (p, k))
            for k in (1, 2)] for p in 'LR']
    ts = os.path.join(GSB, 'sample_gsb_phased.timestamp')

    def fh_open():
        fh = bb.gsb.open(ts, 'rs', raw=raw, sample_rate=1e8 / 3 / 2 ** 19,
                         payload_nbytes=8192, chunk_nbytes=2 * 4 * 8192)
        fh.seek(16)
        return fh

    counts, _ = _check_against_moments(fh_open, samples_per_bin=3 * 16,
                                       count=4 * 16)
    assert counts.shape == (2, 2, 512, 2, 256)
    frames = OUT['gsb_phased_8192_frames'].reshape(-1, 2, 512)[16:80]
    parts = np.stack([frames.real, frames.imag], -1).astype(np.int64)
    assert np.array_equal(counts, _bincount_rows(parts & 0xff, 48))


def refusals():
    from baseband_b200 import tasks
    with bb.dada.open(sample_path('sample_mkbf.dada'), 'rs') as fh:
        with pytest.raises(NotImplementedError):
            tasks.state_counts(fh)


CASES = [vdif_mwa_sample, vdif_synthetic_8bit, guppi_files, guppi_synthetic,
         dada_files, gsb_phased, refusals]


# ------------------------------------------------------------- sharding
def shard_worker(rank, world, port, results, here, use_cpu):
    """One rank of a gloo run of parallel.state_counts_sharded on an 8-bit
    VDIF stream, against the single-process counts."""
    import sys
    sys.path.insert(0, here)
    sys.path.insert(0, os.path.dirname(here))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port),
                      RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    patch = None
    if use_cpu:
        from _pytest.monkeypatch import MonkeyPatch
        patch = MonkeyPatch()
        install(patch)
    import baseband_b200 as bbm
    from baseband_b200 import parallel, synthetic as syn, tasks
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        raw = syn.vdif_stream(6, 4, 1024, bps=8, nchan=2, complex_data=True,
                              seed=31, invalid=[5])
        dev = 'cpu' if use_cpu else 'cuda:0'
        fh = bbm.vdif.open(io.BytesIO(raw.tobytes()), 'rs', sample_rate=1e6,
                           device=dev)
        spf = fh.samples_per_frame
        single = tasks.state_counts(fh, spf)
        ok = single.shape == (6, 4, 2, 2, 256)
        for per_bin in (spf, 4 * spf):
            fh.seek(0)
            counts, (b0, b1) = parallel.state_counts_sharded(fh, per_bin)
            nbin = 6 * spf // per_bin
            ok = ok and (b0, b1) == parallel.shard_bounds(nbin, rank, world)
            ok = ok and np.array_equal(
                counts, single[:nbin * (per_bin // spf)].reshape(
                    (nbin, -1) + single.shape[1:]).sum(1))
        results[rank] = bool(ok)
    finally:
        dist.destroy_process_group()
        if patch is not None:
            patch.undo()


def run_sharded(use_cpu):
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    here = os.path.dirname(os.path.abspath(__file__))
    ctx = mp.get_context('spawn')
    with ctx.Manager() as manager:
        results = manager.dict()
        procs = [ctx.Process(target=shard_worker,
                             args=(r, 2, port, results, here, use_cpu))
                 for r in range(2)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(240)
        assert all(p.exitcode == 0 for p in procs), [p.exitcode
                                                     for p in procs]
        out = dict(results)
    assert out == {0: True, 1: True}


def kernel_case(rng, nelem, nthread, dist, nset=None, unit_bytes=None):
    """A random geometry for bb_byte_counts: shuffled units, some invalid,
    headers of 0 / 4 / 16 bytes (some units not 16-byte aligned), bins that
    cut the call."""
    if unit_bytes is None:
        nsamp = int(rng.integers(1, 600)) * max(1, 4 // nelem)
        unit_bytes = nsamp * nelem
        unit_bytes += (-unit_bytes) % 4
    if nset is None:
        nset = int(rng.integers(1, 6))
    hdr = int(rng.choice([0, 4, 16]))
    frame = unit_bytes + hdr
    nunit = nset * nthread
    n = nunit * frame + 16
    if dist == 'uniform':
        raw = rng.integers(0, 256, n, dtype=np.uint8)
    elif dist == 'one':
        raw = np.full(n, int(rng.integers(0, 256)), np.uint8)
    elif dist == 'two':
        raw = rng.choice(np.array([3, 250], np.uint8), n)
    else:                                             # narrow Gaussian
        raw = np.round(rng.normal(0, 2, n)).astype(np.int64).astype(np.uint8)
    uo = rng.permutation(nunit).astype(np.int64) * frame + hdr
    uo[rng.random(nunit) < 0.15] = -1
    per_bin = int(rng.integers(1, nset + 2))
    origin = int(rng.integers(0, 4))
    nbin = (origin + nset - 1) // per_bin + 1
    return dict(raw=raw, uo=uo, nset=nset, nthread=nthread,
                payload=unit_bytes, nelem=nelem, origin=origin,
                per_bin=per_bin, shape=(nbin, nthread, nelem, 256))


def kernel_want(c):
    want = torch.zeros(c['shape'], dtype=torch.int64)
    byte_counts(torch.from_numpy(c['raw']), torch.from_numpy(c['uo']),
                c['nset'], c['nthread'], c['payload'], c['nelem'], want,
                c['origin'], c['per_bin'])
    return want
