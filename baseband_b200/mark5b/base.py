"""Mark 5B file and stream readers/writers (API of baseband/mark5b/base.py).

Stream reads are batched on the GPU: ``bb_mark5b_scan`` parses all headers of
a chunk (bit fields + BCD) and decides validity from the payload fill pattern;
``bb_decode_bitfield`` then unpacks every payload to ``(nsample, nchan)`` with
invalid frames replaced by ``fill_value``.
"""
import numpy as np
import torch

from .. import kernels, levels
from ..base.opener import make_opener
from ..base.stream import StreamReaderBase, StreamWriterBase, as_hertz
from ..base.utils import bcd_encode, crc_array, crc_remainder
from ..vdif.base import _FileBase
from .frame import Mark5BFrame, FILL_PATTERN
from .header import Mark5BHeader, CRC16
from .payload import Mark5BPayload

__all__ = ['Mark5BFileReader', 'Mark5BFileWriter', 'Mark5BStreamReader',
           'Mark5BStreamWriter', 'open']


class Mark5BFileReader(_FileBase):
    def __init__(self, fh_raw, kday=None, ref_time=None, nchan=None, bps=2):
        super().__init__(fh_raw)
        self.kday, self.ref_time, self.nchan, self.bps = (kday, ref_time,
                                                          nchan, bps)

    def read_header(self):
        return Mark5BHeader.fromfile(self.fh_raw, kday=self.kday,
                                     ref_time=self.ref_time)

    def read_frame(self, verify=True):
        if self.nchan is None:
            raise TypeError('In order to read frames, the file handle '
                            'should be initialized with nchan set.')
        return Mark5BFrame.fromfile(self.fh_raw, kday=self.kday,
                                    ref_time=self.ref_time, nchan=self.nchan,
                                    bps=self.bps, verify=verify)

    def get_frame_rate(self):
        """Highest frame number within a second, plus one
        (base/base.py:371-406)."""
        with self.temporary_offset(0):
            header = self.read_header()
            frame_nr0 = header['frame_nr']
            while header['frame_nr'] == frame_nr0:
                self.fh_raw.seek(10000, 1)
                header = self.read_header()
            highest = frame_nr0
            while header['frame_nr'] > 0:
                highest = max(highest, header['frame_nr'])
                self.fh_raw.seek(10000, 1)
                header = self.read_header()
        return float(highest + 1)

    def _default_pattern(self):
        # the sync word starts every frame (mark5b/header.py:60-63)
        return [0xABADDEED], {'frame_nbytes': 10016}

    def locate_frame(self, maximum=None):
        """Offset of the first sync pattern that is followed by another one a
        frame ahead (or the end of file) and has a correct CRC
        (mark5b/base.py:95-155, forward search only)."""
        start = self.fh_raw.tell()
        size = self.fh_raw.seek(0, 2)
        maximum = 10016 if maximum is None else maximum
        self.fh_raw.seek(start)
        block = np.frombuffer(self.fh_raw.read(maximum + 10016 + 16),
                              np.uint8)
        sync = np.array([0xED, 0xDE, 0xAD, 0xAB], np.uint8)
        hits = np.flatnonzero((block[:-3] == sync[0]) & (block[1:-2] == sync[1])
                              & (block[2:-1] == sync[2])
                              & (block[3:] == sync[3]))
        for h in hits:
            if h > maximum:
                break
            nxt = h + 10016
            if start + nxt + 4 <= size and nxt + 4 <= block.size \
                    and not np.array_equal(block[nxt:nxt + 4], sync):
                continue
            w = block[h:h + 16].copy().view('<u4')
            message = (int(w[2]) << 32) | int(w[3])
            if crc_remainder(message, CRC16, extend=False) == 0:
                self.fh_raw.seek(start + int(h))
                return start + int(h)
        self.fh_raw.seek(start)
        return None


class Mark5BFileWriter(_FileBase):
    def write_frame(self, data, header=None, bps=2, valid=True, **kwargs):
        if not isinstance(data, Mark5BFrame):
            data = Mark5BFrame.fromdata(data, header, bps=bps, valid=valid,
                                        **kwargs)
        return data.tofile(self.fh_raw)


class _Mark5BStreamBase:
    def _get_index(self, header):
        # mark5b/base.py:206-213
        h0 = self.header0
        return int(round(self._frame_rate * (
            header.seconds - h0.seconds
            + 86400 * (header.kday + header.jday - h0.kday - h0.jday))
            + header['frame_nr'] - h0['frame_nr']))

    def _get_time(self, header):
        return header.get_time(frame_rate=self._frame_rate)

    def _set_time(self, header, time):
        header.update(time=time, frame_rate=self._frame_rate)


class Mark5BStreamReader(_Mark5BStreamBase, StreamReaderBase):
    """Mark 5B stream reader (GPU decode).  ``nchan`` is required; ``kday``
    or ``ref_time`` complete the header time."""
    _sample_shape_maker = Mark5BPayload._sample_shape_maker

    def __init__(self, fh_raw, sample_rate=None, kday=None, ref_time=None,
                 nchan=None, bps=2, squeeze=True, subset=(), fill_value=0.,
                 verify=True, device=None, chunk_nbytes=None, dtype=None):
        if nchan is None:
            raise TypeError('Mark 5B stream reader requires nchan to be '
                            'passed in explicitly.')
        fh_raw = Mark5BFileReader(fh_raw, kday=kday, ref_time=ref_time,
                                  nchan=nchan, bps=bps)
        fh_raw.seek(0)
        offset0 = fh_raw.locate_frame()
        if offset0 is None:
            raise OSError('could not find a Mark 5B frame header.')
        self._file_offset0 = offset0
        header0 = fh_raw.read_header()
        sample_rate = as_hertz(sample_rate)
        spf = 10000 * 8 // (bps * nchan)
        if sample_rate is None:
            fh_raw.seek(offset0)
            with fh_raw.temporary_offset(offset0):
                # frame-rate scan starts from the first frame found
                rate = _scan_frame_rate(fh_raw, offset0)
            sample_rate = rate * spf
        size = fh_raw.seek(0, 2)
        self._nframe = (size - offset0) // 10016
        super().__init__(
            fh_raw, header0, sample_rate=sample_rate, samples_per_frame=spf,
            sample_shape=(nchan,), bps=bps, complex_data=False,
            squeeze=squeeze, subset=subset, fill_value=fill_value,
            verify=verify, device=device, chunk_nbytes=chunk_nbytes,
            dtype=dtype)
        self._levels = levels.mark5b(bps)
        self._checks = []
        if self.verify and self._nframe > 1:
            # time of the last frame must match its position, else frames
            # were lost: index all headers
            fh_raw.seek(offset0 + (self._nframe - 1) * 10016)
            try:
                lossy = self._get_index(fh_raw.read_header()) != (
                    self._nframe - 1)
            except Exception:
                lossy = True
            if lossy:
                self._build_index()

    _frame_nbytes = 10016

    def _decode_chunk(self, raw, frame0, nframe, sample_start, nsample, out):
        uo, nthread, payload_nbytes, bps, nelem = self._packed_units(
            raw, frame0, nframe)
        kernels.decode_bitfield(
            raw, uo, nframe, nthread, payload_nbytes, bps, nelem, False,
            kernels.CODEC_LEVELS, self._levels, self._fill_value,
            sample_start, nsample, out)

    def _packed_units(self, raw, frame0, nframe):
        if self._index is not None:
            # irregular stream: the frames of the chunk sit where the index
            # says (`_chunk_layout`); the scan still decides payload validity
            rel = self._chunk_layout(frame0, nframe)[4][:, 0]
            _, uo = kernels.mark5b_scan(
                raw, nframe, frame_offset=torch.from_numpy(
                    np.ascontiguousarray(rel)).to(raw.device),
                want_fields=False)
        else:
            # with verify, the frame index the header time implies
            # (mark5b/base.py:206-213) is checked inside the scan kernel
            h0 = self.header0
            check = ((frame0, h0.jday, h0.seconds, h0['frame_nr'],
                      int(round(self._frame_rate))) if self.verify else None)
            _, uo = kernels.mark5b_scan(
                raw, nframe, check=check,
                bad=self._bad_counter(raw.device) if self.verify else None,
                want_fields=False)
        return uo, 1, 10000, self._bps, self._sample_shape[0]

    def _frame_index(self, jday, seconds, frame_nr):
        """mark5b/base.py:206-213 on arrays (torch or numpy); jday wraps
        every 1000 days."""
        h0 = self.header0
        fps = int(round(self._frame_rate))
        dday = (jday - h0.jday + 500) % 1000 - 500
        return ((seconds - h0.seconds + 86400 * dday) * fps
                + frame_nr - h0['frame_nr'])

    def _build_index(self):
        """Frame table of a stream with missing / duplicated / re-ordered
        frames or bytes lost between frames, built on the GPU from every sync
        word 0xABADDEED that is followed by another one a frame later (cf.
        VDIFStreamReader._build_index)."""
        h0 = self.header0
        size = self.fh_raw.seek(0, 2)
        self.fh_raw.seek(0)
        nphys = (size - self._file_offset0) // 10016
        fps = int(round(self._frame_rate))
        nset_max = 2 * nphys + fps + 2

        def index_chunk(raw, base, locations, count, table, stats):
            kernels.mark5b_index(raw, base, locations, count, h0.jday,
                                 h0.seconds, h0['frame_nr'], fps, nset_max,
                                 table, stats)

        table, stats = self._build_index_on_device(
            [0xABADDEED], [0xffffffff], 10016, index_chunk, 1, nset_max)
        # (headers whose BCD time code cannot be read are not placed: their
        # frames read as fill_value, as in the reference's repair)
        self._set_index_table(table, 10016)

    def read(self, count=None, out=None, **kwargs):
        offset = self.offset
        result = super().read(count, out, **kwargs)
        if self._index is None and self._new_inconsistencies():
            if not self.verify:
                raise OSError('Mark 5B stream is not a regular sequence of '
                              'frames and verify is off.')
            import warnings
            warnings.warn('Mark 5B stream has missing or out-of-order '
                          'frames; indexing all headers and filling the '
                          'gaps with fill_value.')
            self._build_index()
            self.offset = offset
            return super().read(None if count is None and out is None
                                else result.shape[0], out, **kwargs)
        return result


def _scan_frame_rate(fh_raw, offset0):
    fh = fh_raw.fh_raw
    fh.seek(offset0)
    header = fh_raw.read_header()
    frame_nr0 = header['frame_nr']
    while header['frame_nr'] == frame_nr0:
        fh.seek(10000, 1)
        header = fh_raw.read_header()
    highest = frame_nr0
    while header['frame_nr'] > 0:
        highest = max(highest, header['frame_nr'])
        fh.seek(10000, 1)
        header = fh_raw.read_header()
    return float(highest + 1)


class Mark5BStreamWriter(_Mark5BStreamBase, StreamWriterBase):
    """Mark 5B stream writer (GPU encode)."""
    _sample_shape_maker = Mark5BPayload._sample_shape_maker

    def __init__(self, fh_raw, header0=None, sample_rate=None, nchan=1,
                 bps=2, squeeze=True, device=None):
        fh_raw = Mark5BFileWriter(fh_raw)
        spf = 10000 * 8 // (bps * nchan)
        super().__init__(fh_raw, header0, sample_rate=sample_rate,
                         samples_per_frame=spf, sample_shape=(nchan,),
                         bps=bps, complex_data=False, squeeze=squeeze,
                         device=device)

    def _encode_frames(self, flat, index0, nframe, valid):
        h0 = self.header0
        dev = flat.device
        fps = int(round(self._frame_rate))
        # header words per frame: mark5b/base.py:215-225 (_set_index)
        index = np.arange(index0, index0 + nframe, dtype=np.int64)
        dt, frame_nr = np.divmod(index + h0['frame_nr'], fps)
        seconds = h0.seconds + dt
        dday, seconds = np.divmod(seconds, 86400)
        jday = (h0.jday + dday) % 1000
        # fraction: ns rounded, then truncated to 0.1 ms (header.py:223-230)
        ns = np.round(frame_nr / self._frame_rate * 1e9).astype(np.int64)
        frac = ns // 100000
        bj, bs, bf = bcd_encode(jday), bcd_encode(seconds), bcd_encode(frac)
        words = np.empty((nframe, 4), np.uint32)
        words[:, 0] = h0.words[0]
        words[:, 1] = ((np.uint32(h0.words[1]) & np.uint32(0xffff8000))
                       | frame_nr.astype(np.uint32))
        words[:, 2] = ((bj << 20) | bs).astype(np.uint32)
        stream = (((bj << 20) | bs) << 16) | bf
        crc = crc_array(stream, 48, CRC16)
        words[:, 3] = ((bf << 16) | crc).astype(np.uint32)
        # headers into place, unit offsets, and -- for invalid frames -- the
        # fill pattern instead of an encoded payload (mark5b/frame.py:126-133)
        # in one launch; the encode skips units at -1
        frames, uo = kernels.frames_assemble(
            torch.from_numpy(words.view(np.uint8)).to(dev), 10016, 10000,
            valid=None if valid.all() else torch.from_numpy(
                valid.astype(np.uint8)).to(dev), fill_word=FILL_PATTERN)
        kernels.encode_bitfield(flat, frames.view(-1), uo, nframe, 1,
                                10000, self._bps, self._sample_shape[0],
                                kernels.QUANT_MARK5B)
        return frames.view(-1)


open = make_opener('mark5b', {'rb': Mark5BFileReader, 'wb': Mark5BFileWriter,
                              'rs': Mark5BStreamReader,
                              'ws': Mark5BStreamWriter},
                   header_class=Mark5BHeader,
                   non_header_keys={'sample_rate', 'nchan', 'bps', 'kday',
                                    'ref_time'},
                   doc="""Open Mark 5B file(s) for reading or writing.

Reader options: ``sample_rate``, ``kday`` or ``ref_time``, ``nchan``
(required), ``bps``, ``squeeze``, ``subset``, ``fill_value``, ``verify``,
``device``.  Writer: ``header0`` or header keywords (``time=...``),
``sample_rate``, ``nchan``, ``bps``, ``squeeze``, ``device``.
""")
