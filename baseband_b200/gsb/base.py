"""GSB stream reader/writer (API of baseband/gsb/base.py): a timestamp text
file plus one raw file (rawdump) or ``raw[pol][part]`` files (phased).

For a range of frames the reader copies the matching byte range of every raw
file into one pinned buffer; the unit table of ``bb_decode_bitfield`` (one
unit per frame, part and polarisation) then expresses the part/polarisation
interleave of gsb/payload.py:115-131, so the decode kernel assembles
``(nsample, npol, nchan)`` directly.
"""
import io
import os

import numpy as np
import torch

from .. import kernels
from ..base.opener import normalize_mode
from ..base.stream import (StreamReaderBase, StreamWriterBase, as_hertz,
                           read_file_into)
from ..vdif.base import _FileBase
from .frame import GSBFrame
from .header import GSBHeader
from .payload import GSBPayload

__all__ = ['GSBTimeStampIO', 'GSBFileReader', 'GSBFileWriter',
           'GSBStreamReader', 'GSBStreamWriter', 'open']

DEFAULT_FRAME_RATE = 1e8 / 6 / 2 ** 22        # 0.25165824 s per frame


class GSBTimeStampIO(_FileBase):
    def read_timestamp(self):
        return GSBHeader.fromfile(self.fh_raw)

    def write_timestamp(self, header=None, **kwargs):
        if header is None:
            header = GSBHeader.fromvalues(**kwargs)
        return header.tofile(self.fh_raw)


class GSBFileReader(_FileBase):
    def __init__(self, fh_raw, payload_nbytes=None, nchan=None, bps=None,
                 complex_data=None):
        super().__init__(fh_raw)
        self.payload_nbytes, self.nchan, self.bps, self.complex_data = (
            payload_nbytes, nchan, bps, complex_data)

    def read_payload(self):
        return GSBPayload.fromfile(
            self.fh_raw, payload_nbytes=self.payload_nbytes,
            sample_shape=(self.nchan,), bps=self.bps,
            complex_data=self.complex_data)


class GSBFileWriter(_FileBase):
    def write_payload(self, data, bps=4):
        if not isinstance(data, GSBPayload):
            data = GSBPayload.fromdata(data, bps=bps)
        return data.tofile(self.fh_raw)


def _geometry(header0, fh_raw, sample_rate, samples_per_frame,
              payload_nbytes, nchan, bps, complex_data):
    """Defaults and consistency of gsb/base.py:146-201."""
    rawdump = header0.mode == 'rawdump'
    if isinstance(fh_raw, (tuple, list)):
        assert not rawdump
        if not isinstance(fh_raw[0], (tuple, list)):
            fh_raw = (tuple(fh_raw),)
        for pair in fh_raw:
            assert len(pair) == len(fh_raw[0])
    elif not rawdump:
        fh_raw = ((fh_raw,),)
    complex_data = (not rawdump) if complex_data is None else complex_data
    bps = (4 if rawdump else 8) if bps is None else bps
    nchan = (1 if rawdump else 512) if nchan is None else nchan
    bpfs = bps * nchan * (2 if complex_data else 1)
    nfiles = 1 if rawdump else len(fh_raw[0])
    sample_rate = as_hertz(sample_rate)
    if payload_nbytes is None:
        if samples_per_frame is None:
            payload_nbytes = (2 ** 22 if sample_rate is None else int(round(
                sample_rate / DEFAULT_FRAME_RATE * bpfs / 8 / nfiles)))
        else:
            payload_nbytes = samples_per_frame * bpfs // (8 * nfiles)
    if samples_per_frame is None:
        samples_per_frame = payload_nbytes * 8 // bpfs * nfiles
    elif samples_per_frame != payload_nbytes * nfiles * 8 / bpfs:
        raise ValueError('inconsistent samples_per_frame, bps, complex_data, '
                         'and payload_nbytes')
    if sample_rate is None:
        sample_rate = samples_per_frame * DEFAULT_FRAME_RATE
    sample_shape = (nchan,) if rawdump else (len(fh_raw), nchan)
    return dict(fh_raw=fh_raw, sample_rate=sample_rate,
                samples_per_frame=samples_per_frame,
                payload_nbytes=payload_nbytes, sample_shape=sample_shape,
                bps=bps, complex_data=complex_data, nfiles=nfiles)


class _GSBStreamBase:
    _sample_shape_maker = staticmethod(GSBPayload._sample_shape_maker)

    def _files(self):
        if self.header0.mode == 'rawdump':
            return [[self.fh_raw]]
        return self.fh_raw

    @property
    def payload_nbytes(self):
        return self._payload_nbytes

    def close(self):
        self._closed = True
        self.fh_ts.close()
        for group in self._files():
            for fh in group:
                fh.close()

    @property
    def closed(self):
        return self._closed

    @property
    def name(self):
        return getattr(self.fh_ts, 'name', None)


class GSBStreamReader(_GSBStreamBase, StreamReaderBase):
    """GSB stream reader (GPU decode)."""

    def __init__(self, fh_ts, fh_raw, sample_rate=None,
                 samples_per_frame=None, payload_nbytes=None, nchan=None,
                 bps=None, complex_data=None, squeeze=True, subset=(),
                 verify=True, device=None, chunk_nbytes=None, dtype=None):
        self.fh_ts = GSBTimeStampIO(fh_ts)
        header0 = self.fh_ts.read_timestamp()
        g = _geometry(header0, fh_raw, sample_rate, samples_per_frame,
                      payload_nbytes, nchan, bps, complex_data)
        self._payload_nbytes = g['payload_nbytes']
        self._nfiles = g['nfiles']
        super().__init__(
            g['fh_raw'], header0, sample_rate=g['sample_rate'],
            samples_per_frame=g['samples_per_frame'],
            sample_shape=g['sample_shape'], bps=g['bps'],
            complex_data=g['complex_data'], squeeze=squeeze, subset=subset,
            verify=verify, device=device, chunk_nbytes=chunk_nbytes,
            dtype=dtype)
        # frames = complete timestamp lines that also have payload bytes
        self.fh_ts.seek(0)
        text = self.fh_ts.read()
        if isinstance(text, bytes):
            text = text.decode('ascii')
        lines = [ln for ln in text.split('\n')]
        nwords = len(header0.words)
        nline = 0
        for ln in lines:
            if len(ln.split()) != nwords:
                break
            nline += 1
        sizes = []
        for group in self._files():
            for fh in group:
                pos = fh.tell()
                sizes.append(fh.seek(0, 2) // self._payload_nbytes)
                fh.seek(pos)
        self._nframe = min([nline] + sizes)

    @property
    def _frame_nbytes(self):
        files = self._files()
        return self._payload_nbytes * len(files) * len(files[0])

    def _read_raw(self, frame0, nframe, pinned, sample_start=0, nsample=0):
        view = pinned.numpy()
        span = nframe * self._payload_nbytes
        k = 0
        for group in self._files():
            for fh in group:
                got = read_file_into(fh, frame0 * self._payload_nbytes,
                                     view[k * span:(k + 1) * span])
                if got != span:
                    raise EOFError('could not read {} frames at frame {}.'
                                   .format(nframe, frame0))
                k += 1

    def _decode_chunk(self, raw, frame0, nframe, sample_start, nsample, out):
        uo, npol, pn, bps, nelem, npart = self._packed_units(raw, frame0,
                                                             nframe)
        kernels.decode_bitfield(
            raw, uo, nframe * npart, npol, pn, bps, nelem, self._complex_data,
            kernels.CODEC_SINT, None, self._fill_value, sample_start, nsample,
            out)

    def _packed_units(self, raw, frame0, nframe):
        """Unit table of a chunk (the raw files' pieces sit one after the
        other in ``raw``, `_read_raw`): a frame is ``npart`` sets of ``npol``
        units (`tasks.state_counts` for the 4-bit modes, `tasks.moments` for
        8 bit)."""
        files = self._files()
        npol, npart = len(files), len(files[0])
        pn = self._payload_nbytes
        span = nframe * pn
        frame = np.arange(nframe, dtype=np.int64)[:, None, None]
        part = np.arange(npart, dtype=np.int64)[None, :, None]
        pol = np.arange(npol, dtype=np.int64)[None, None, :]
        uo = ((pol * npart + part) * span + frame * pn).reshape(-1)
        nchan = self._sample_shape[-1]
        nelem = nchan * (2 if self._complex_data else 1)
        return (torch.from_numpy(uo).to(raw.device), npol, pn, self._bps,
                nelem, npart)

    @property
    def _levels(self):
        """Value of every 4-bit code (two's complement nibbles,
        gsb/payload.py:19-42), for `tasks.state_levels`; 8-bit streams are
        summarised by their moments instead."""
        if self._bps != 4:
            return None
        code = np.arange(16)
        return np.where(code < 8, code, code - 16).astype(np.float32)

    def _moments_view(self, m):
        """(nbin, npol, nchan * parts, 3) -> (nbin,) + sample shape + parts."""
        ib = 2 if self._complex_data else 1
        m = m.reshape((m.shape[0],) + tuple(self._sample_shape) + (ib, 3))
        return m if ib == 2 else m[..., 0, :]


class GSBStreamWriter(_GSBStreamBase, StreamWriterBase):
    """GSB stream writer (GPU encode)."""

    def __init__(self, fh_ts, fh_raw, header0=None, sample_rate=None,
                 samples_per_frame=None, payload_nbytes=None, nchan=None,
                 bps=None, complex_data=None, squeeze=True, device=None,
                 **kwargs):
        if 'dtype' in kwargs:
            # as for the other formats' writers: `dtype` is a reader option
            raise TypeError("GSBStreamWriter got an unexpected keyword "
                            "argument 'dtype'")
        self.fh_ts = GSBTimeStampIO(fh_ts)
        if header0 is None:
            header0 = GSBHeader.fromvalues(**kwargs)
        g = _geometry(header0, fh_raw, sample_rate, samples_per_frame,
                      payload_nbytes, nchan, bps, complex_data)
        self._payload_nbytes = g['payload_nbytes']
        super().__init__(
            g['fh_raw'], header0, sample_rate=g['sample_rate'],
            samples_per_frame=g['samples_per_frame'],
            sample_shape=g['sample_shape'], bps=g['bps'],
            complex_data=g['complex_data'], squeeze=squeeze, device=device)

    def _set_index(self, header, index):
        from fractions import Fraction
        dt = Fraction(index) / Fraction(self._frame_rate).limit_denominator(
            10**12)
        if self.header0.mode == 'phased':
            header.update(gps_time=self.header0.gps_time + dt,
                          pc_time=self.header0.pc_time + dt,
                          seq_nr=self.header0['seq_nr'] + index,
                          mem_block=(self.header0['mem_block'] + index) % 8)
        else:
            header.update(time=self.header0.time + dt)

    def _encode_frames(self, flat, index0, nframe, valid):
        files = self._files()
        npol, npart = len(files), len(files[0])
        pn = self._payload_nbytes
        span = nframe * pn
        dev = flat.device
        frame = np.arange(nframe, dtype=np.int64)[:, None, None]
        part = np.arange(npart, dtype=np.int64)[None, :, None]
        pol = np.arange(npol, dtype=np.int64)[None, None, :]
        uo = ((pol * npart + part) * span + frame * pn).reshape(-1)
        packed = torch.empty(npol * npart * span, dtype=torch.uint8,
                             device=dev)
        nelem = self._sample_shape[-1] * (2 if self._complex_data else 1)
        kernels.encode_bitfield(flat, packed, torch.from_numpy(uo).to(dev),
                                nframe * npart, npol, pn, self._bps, nelem,
                                kernels.QUANT_SINT)
        self._header_lines = []
        for i in range(nframe):
            header = self.header0.copy()
            header.mutable = True
            self._set_index(header, index0 + i)
            self._header_lines.append(header)
        return packed

    def _write_raw(self, frames):
        from .. import device as _device
        host = _device.pinned_empty(frames.shape, torch.uint8)
        host.copy_(frames, non_blocking=True)
        _device.current_stream_synchronize(frames.device)
        files = self._files()
        span = host.numel() // (len(files) * len(files[0]))
        view = host.numpy()
        k = 0
        for group in files:
            for fh in group:
                fh.write(memoryview(view[k * span:(k + 1) * span]))
                k += 1
        for header in self._header_lines:
            header.tofile(self.fh_ts.fh_raw)


def open(name, mode='rs', **kwargs):
    """Open GSB file(s).  ``name`` is the timestamp file; ``raw`` the raw
    data file (rawdump) or nested tuple ``raw[pol][part]`` (phased).  Modes:
    'rt'/'wt' timestamp file only, 'rb'/'wb' one raw file, 'rs'/'ws' streams.
    Stream options: ``sample_rate``, ``samples_per_frame`` or
    ``payload_nbytes``, ``nchan``, ``bps``, ``complex_data``, ``squeeze``,
    ``subset``, ``verify``, ``device``; writers take ``header0`` or header
    keywords (``time``, and for phased ``seq_nr``, ``mem_block``...)."""
    if mode in ('rt', 'wt'):
        fh = io.open(name, mode) if isinstance(
            name, (str, bytes, os.PathLike)) else name
        return GSBTimeStampIO(fh)
    mode = normalize_mode(mode)

    def _open(f, m):
        return io.open(f, m) if isinstance(f, (str, bytes, os.PathLike)) else f

    if mode[1] == 'b':
        cls = GSBFileReader if mode[0] == 'r' else GSBFileWriter
        return cls(_open(name, mode), **kwargs)
    raw = kwargs.pop('raw')
    fh_ts = _open(name, mode[0] + 't')
    if isinstance(raw, (tuple, list)):
        if not isinstance(raw[0], (tuple, list)):
            raw = (tuple(raw),)
        fh_raw = tuple(tuple(_open(f, mode[0] + 'b') for f in group)
                       for group in raw)
    else:
        fh_raw = _open(raw, mode[0] + 'b')
    cls = GSBStreamReader if mode[0] == 'r' else GSBStreamWriter
    return cls(fh_ts, fh_raw, **kwargs)
