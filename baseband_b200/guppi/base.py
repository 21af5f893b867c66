"""GUPPI file and stream readers/writers (API of baseband/guppi/base.py).

Stream reads honour the overlap rule of the reference exactly
(guppi/base.py:203-221, :270-278 with the generic loop at
base/base.py:957-967): the stream advances ``samples_per_frame - overlap``
samples per frame; a read takes ``[start, len)`` from the frame it starts in
and ``[overlap, len)`` from every later frame, where ``len`` includes the
overlap.  These per-frame windows become the ``col_begin / col_end /
out_col0`` tables of one ``bb_decode_int8_transposed`` launch per chunk.
"""
import numpy as np

from ..base.opener import make_opener
from ..base.stream import StreamReaderBase, StreamWriterBase
from ..vdif.base import _FileBase
from .frame import GUPPIFrame
from .header import GUPPIHeader
from .payload import GUPPIPayload, decode_device

__all__ = ['GUPPIFileReader', 'GUPPIFileWriter', 'GUPPIStreamReader',
           'GUPPIStreamWriter', 'open']


class GUPPIFileReader(_FileBase):
    def read_header(self):
        return GUPPIHeader.fromfile(self.fh_raw)

    def read_frame(self, memmap=True, verify=True):
        return GUPPIFrame.fromfile(self.fh_raw, memmap=memmap, verify=verify)

    def get_frame_rate(self):
        with self.temporary_offset(0):
            header = self.read_header()
        return (header.sample_rate
                / (header.samples_per_frame - header.overlap))


class GUPPIFileWriter(_FileBase):
    def write_frame(self, data, header=None, **kwargs):
        if not isinstance(data, GUPPIFrame):
            data = GUPPIFrame.fromdata(data, header, **kwargs)
        return data.tofile(self.fh_raw)

    def memmap_frame(self, header=None, **kwargs):
        """Write the header now and map the payload, so that the frame can
        be filled in pieces by assigning to slices of it
        (guppi/base.py:169-192)."""
        if header is None:
            header = GUPPIHeader.fromvalues(**kwargs)
        header.tofile(self.fh_raw)
        payload = GUPPIPayload.fromfile(self.fh_raw, memmap=True,
                                        header=header)
        return GUPPIFrame(header, payload)


class _GUPPIStreamBase:
    _sample_shape_maker = GUPPIPayload._sample_shape_maker

    @property
    def _packets_per_frame(self):
        h0 = self.header0
        return ((h0.payload_nbytes - h0.overlap * h0._bpcs // 8)
                // int(h0['PKTSIZE']))

    def _get_index(self, header):
        return int(round((header['PKTIDX'] - self.header0['PKTIDX'])
                         / self._packets_per_frame))

    def _set_index(self, header, index):
        header.update(pktidx=self.header0['PKTIDX']
                      + index * self._packets_per_frame)


class GUPPIStreamReader(_GUPPIStreamBase, StreamReaderBase):
    """GUPPI stream reader (GPU decode).  ``samples_per_frame`` excludes the
    overlap."""

    def __init__(self, fh_raw, squeeze=True, subset=(), verify=True,
                 device=None, chunk_nbytes=None, dtype=None):
        fh_raw = GUPPIFileReader(fh_raw)
        header0 = fh_raw.read_header()
        self._full_spf = header0.samples_per_frame
        self._overlap = header0.overlap
        self._small_read_cache_ok = self._overlap == 0
        self._frame_nbytes = header0.frame_nbytes
        size = fh_raw.seek(0, 2)
        self._nframe = size // header0.frame_nbytes
        super().__init__(
            fh_raw, header0, squeeze=squeeze, subset=subset, verify=verify,
            samples_per_frame=self._full_spf - self._overlap,
            device=device, chunk_nbytes=chunk_nbytes, dtype=dtype)

    @property
    def _nsample(self):
        return self._nframe * self._samples_per_frame + self._overlap

    def _locate(self, offset):
        """Frame and frame-local sample of stream sample ``offset``."""
        stride = self._samples_per_frame
        normal_end = self._nsample - self._overlap
        if normal_end <= offset < self._nsample:   # overlap of last frame
            return self._nframe - 1, stride + offset - normal_end
        return divmod(offset, stride)

    def _chunks(self, start, count):
        """(frame0, nframe, local start in frame0, nsample, row0).  Frames
        after the one a read starts in contribute from ``overlap`` on."""
        if count == 0:
            return
        full = self._full_spf
        frame, local = self._locate(start)
        per = self._frames_per_chunk()
        row = 0
        while row < count:
            nframe, n, first = 0, 0, local
            while nframe < per and row + n < count and \
                    frame + nframe < self._nframe:
                n += min(full - local, count - row - n)
                nframe += 1
                local = self._overlap
            yield frame, nframe, first, n, row
            frame += nframe
            row += n

    def _packed_units(self, raw, frame0, nframe):
        """Units for consumers that work on the packed int8 samples
        (`tasks.moments`): the non-overlap part of every frame.  Channels
        first: one unit per channel row (`thread` = channel, elements = pol x
        (re, im)); time first: one unit per frame (elements = chan x pol x
        (re, im))."""
        import torch
        h0 = self.header0
        if h0.bps != 8:
            raise KeyError(h0.bps)
        ib = 2 if h0.complex_data else 1
        spf = self._samples_per_frame                  # without the overlap
        start = np.arange(nframe, dtype=np.int64) * self._frame_nbytes \
            + h0.nbytes
        if h0.channels_first:
            rowbytes = self._full_spf * h0.npol * ib
            uo = start[:, None] + np.arange(h0.nchan, dtype=np.int64) \
                * rowbytes
            geom = (h0.nchan, spf * h0.npol * ib, 8, h0.npol * ib)
        else:
            uo = start
            geom = (1, spf * h0.nchan * h0.npol * ib, 8,
                    h0.nchan * h0.npol * ib)
        uo = torch.from_numpy(np.ascontiguousarray(uo.reshape(-1))).to(
            raw.device)
        return (uo,) + geom

    def _decode_chunk(self, raw, frame0, nframe, sample_start, nsample, out):
        h0 = self.header0
        offsets = np.arange(nframe) * self._frame_nbytes + h0.nbytes
        begin = np.full(nframe, self._overlap, np.int64)
        begin[0] = sample_start
        end = np.full(nframe, self._full_spf, np.int64)
        end[-1] -= (end - begin).sum() - nsample
        if h0.bps != 8:
            raise KeyError(h0.bps)
        decode_device(raw, offsets, self._full_spf, h0.npol, h0.nchan,
                      h0.complex_data, h0.channels_first, begin, end,
                      out=out)

    @property
    def stop_time(self):
        return self.start_time + self._offset_seconds(self._nsample)


class GUPPIStreamWriter(_GUPPIStreamBase, StreamWriterBase):
    """GUPPI stream writer (GPU encode); overlap must be 0."""

    def __init__(self, fh_raw, header0, squeeze=True, device=None):
        assert header0.get('OVERLAP', 0) == 0, (
            'overlap must be 0 when writing GUPPI files.')
        fh_raw = GUPPIFileWriter(fh_raw)
        super().__init__(fh_raw, header0, squeeze=squeeze, device=device)

    def _encode_frames(self, flat, index0, nframe, valid):
        import torch
        from .. import kernels
        h0 = self.header0
        dev = flat.device
        hdr_nbytes, frame_nbytes = h0.nbytes, h0.frame_nbytes
        texts = []
        for i in range(nframe):
            header = h0.copy()
            header.mutable = True
            self._set_index(header, index0 + i)
            raw = header.tostring().encode('ascii')
            texts.append(np.frombuffer(
                raw + b'\0' * (hdr_nbytes - len(raw)), np.uint8))
        frames, uo = kernels.frames_assemble(
            torch.from_numpy(np.stack(texts)).to(dev), frame_nbytes)
        spf, ib = self._samples_per_frame, 2 if h0.complex_data else 1
        if h0.bps != 8:
            raise ValueError('GUPPIPayload cannot encode data with {} bits'
                             .format(h0.bps))
        if h0.channels_first:
            kernels.encode_int8_transposed(flat, frames.view(-1), uo, nframe,
                                           h0.nchan, spf * h0.npol, ib)
        else:
            kernels.encode_int8_timefirst(flat, frames.view(-1), uo, nframe,
                                          spf, h0.nchan, h0.npol, ib)
        return frames.view(-1)


open = make_opener('guppi', {'rb': GUPPIFileReader, 'wb': GUPPIFileWriter,
                             'rs': GUPPIStreamReader,
                             'ws': GUPPIStreamWriter},
                   header_class=GUPPIHeader,
                   doc="""Open GUPPI raw file(s) for reading or writing.

Reader options: ``squeeze``, ``subset``, ``verify``, ``device``.  Writer:
``header0`` or header keywords (``time``, ``sample_rate``,
``samples_per_frame``, ``sample_shape`` or ``npol``/``nchan`` ...),
``squeeze``, ``device``.
""")
