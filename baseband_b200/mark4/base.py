"""Mark 4 file and stream readers/writers (API of baseband/mark4/base.py).

A stream read is batched on the GPU: ``bb_mark4_scan`` bit-transposes the
track headers of every frame in a chunk (time code of one track + the error
flags of all tracks -> frame validity) and ``bb_mark4_decode`` undoes the
track/fan-out bit interleave of all payloads, writing ``(nsample, nchan)``
with the header-overwritten samples and invalid frames set to ``fill_value``.
"""
import numpy as np
import torch

from .. import kernels, levels, codecs
from ..base.opener import make_opener
from ..base.stream import StreamReaderBase, StreamWriterBase, as_hertz
from ..base.utils import bcd_encode, crc_of_bits
from ..vdif.base import _FileBase
from .frame import Mark4Frame
from .header import (Mark4Header, stream2words, words2stream, MARK4_DTYPES,
                     CRC12)
from .payload import Mark4Payload

__all__ = ['Mark4FileReader', 'Mark4FileWriter', 'Mark4StreamReader',
           'Mark4StreamWriter', 'open']


class Mark4FileReader(_FileBase):
    """Binary-level reader.  ``ntrack`` may be None, in which case it is
    determined from the spacing of sync patterns."""

    def __init__(self, fh_raw, ntrack=None, decade=None, ref_time=None):
        super().__init__(fh_raw)
        self.ntrack, self.decade, self.ref_time = ntrack, decade, ref_time

    def read_header(self):
        return Mark4Header.fromfile(self.fh_raw, ntrack=self.ntrack,
                                    decade=self.decade,
                                    ref_time=self.ref_time)

    def read_frame(self, verify=True):
        return Mark4Frame.fromfile(self.fh_raw, self.ntrack,
                                   decade=self.decade,
                                   ref_time=self.ref_time, verify=verify)

    def get_frame_rate(self):
        """From the time difference of the first two headers."""
        with self.temporary_offset():
            self.locate_frame()
            h0 = self.read_header()
            self.fh_raw.seek(h0.payload_nbytes, 1)
            h1 = self.read_header()
        dt = h1.time - h0.time
        return float(1 / dt)

    def _default_pattern(self):
        # every track carries the all-ones sync word at steps 64..95
        # (mark4/header.py:125-131)
        if self.ntrack is None:
            raise ValueError('ntrack is needed to locate frames; use '
                             'determine_ntrack() first.')
        nb = self.ntrack // 8
        return np.full(32 * nb, 0xff, np.uint8), {
            'frame_nbytes': self.ntrack * 2500, 'offset': 64 * nb}

    def locate_frame(self, forward=True, maximum=None):
        """Move to the first frame: the byte position where every track has
        the 32-step all-ones sync word at steps 64..95 and again one frame
        later (or the file ends).  Returns the offset or None."""
        ntrack = self.ntrack
        if ntrack is None:
            raise ValueError('ntrack is needed to locate frames; use '
                             'determine_ntrack() first.')
        nset = ntrack // 8                    # bytes per time step
        frame_nbytes = ntrack * 2500
        start = self.fh_raw.tell()
        size = self.fh_raw.seek(0, 2)
        maximum = 2 * frame_nbytes if maximum is None else maximum
        self.fh_raw.seek(start)
        block = np.frombuffer(self.fh_raw.read(maximum + frame_nbytes
                                               + 96 * nset), np.uint8)
        # runs of >= 32*nset bytes of 0xff
        ones = np.concatenate([[0], (block == 0xff).astype(np.int8), [0]])
        edges = np.flatnonzero(np.diff(ones))
        for a, b in zip(edges[::2], edges[1::2]):
            if b - a < 32 * nset:
                continue
            # the sync word may be preceded by set bits of word 1: try each
            # step-aligned candidate in the run
            for s in range(a, b - 32 * nset + 1):
                off = s - 64 * nset
                if off < 0 or off > maximum:
                    continue
                nxt = off + frame_nbytes + 64 * nset
                if start + nxt + 32 * nset <= size:
                    if nxt + 32 * nset > block.size or not np.all(
                            block[nxt:nxt + 32 * nset] == 0xff):
                        continue
                # word 1 lsb (step 63) is always 0: the run must start here
                if s > 0 and np.all(block[s - nset:s] == 0xff):
                    continue
                self.fh_raw.seek(start + off)
                return start + off
        self.fh_raw.seek(start)
        return None

    def determine_ntrack(self, maximum=None):
        """Try ntrack = 16, 32, 64 until frames are found."""
        old = self.ntrack
        for ntrack in (16, 32, 64):
            self.ntrack = ntrack
            with self.temporary_offset():
                if self.locate_frame(maximum=maximum) is not None:
                    try:
                        self.read_header()
                        return ntrack
                    except Exception:
                        pass
        self.ntrack = old
        raise ValueError('cannot determine ntrack automatically.')


class Mark4FileWriter(_FileBase):
    def write_frame(self, data, header=None, **kwargs):
        if not isinstance(data, Mark4Frame):
            data = Mark4Frame.fromdata(data, header, **kwargs)
        return data.tofile(self.fh_raw)


class Mark4StreamReader(StreamReaderBase):
    """Mark 4 stream reader (GPU decode)."""
    _sample_shape_maker = Mark4Payload._sample_shape_maker

    def __init__(self, fh_raw, sample_rate=None, ntrack=None, decade=None,
                 ref_time=None, squeeze=True, subset=(), fill_value=0.,
                 verify=True, device=None, chunk_nbytes=None, dtype=None):
        if decade is None and ref_time is None:
            raise TypeError('Mark 4 stream reader requires either decade or '
                            'ref_time to be passed in.')
        fh_raw = Mark4FileReader(fh_raw, ntrack=ntrack, decade=decade,
                                 ref_time=ref_time)
        fh_raw.seek(0)
        if ntrack is None:
            fh_raw.determine_ntrack()
        offset0 = fh_raw.locate_frame()
        if offset0 is None:
            raise OSError('could not find a Mark 4 frame.')
        self._file_offset0 = offset0
        header0 = fh_raw.read_header()
        sample_rate = as_hertz(sample_rate)
        if sample_rate is None:
            fh_raw.seek(offset0)
            sample_rate = fh_raw.get_frame_rate() * header0.samples_per_frame
        size = fh_raw.seek(0, 2)
        self._frame_nbytes = header0.frame_nbytes
        self._nframe = (size - offset0) // header0.frame_nbytes
        super().__init__(
            fh_raw, header0, sample_rate=sample_rate, squeeze=squeeze,
            subset=subset, fill_value=fill_value, verify=verify,
            device=device, chunk_nbytes=chunk_nbytes, dtype=dtype)
        coder = Mark4Payload(np.zeros(
            header0.payload_nbytes // header0.stream_dtype.itemsize,
            header0.stream_dtype), header0)._coder
        try:
            self._mode = codecs._M4_MODES[coder]
        except KeyError:
            raise KeyError('no Mark 4 decoder for (nchan, bps, fanout) = '
                           '{}'.format(coder))
        self._levels = levels.sign_magnitude()
        self._tick = None
        if self.verify and self._nframe > 1:
            # the time of the last frame must match its position, else frames
            # were lost (or bytes slipped): index the file
            fh_raw.seek(offset0 + (self._nframe - 1) * header0.frame_nbytes)
            try:
                last = fh_raw.read_header()
                lossy = int(round((last.time - header0.time)
                                  * self._frame_rate)) != self._nframe - 1
            except Exception:
                lossy = True
            if lossy:
                self._build_index()

    def _decode_chunk(self, raw, frame0, nframe, sample_start, nsample, out):
        nchan, fanout, ft = self._mode
        uo = self._payload_offsets(raw, frame0, nframe)
        kernels.mark4_decode(raw, uo, nframe, nchan, fanout, ft,
                             self._levels, self._fill_value, sample_start,
                             nsample, out)

    def _count_states(self, raw, frame0, nframe, counts, origin, per_bin):
        """Consumer hook of `tasks.state_counts`: (sign, magnitude) states
        per channel straight from the track words of a chunk; the 160 header
        steps of every frame and invalid frames are not counted."""
        nchan, fanout, ft = self._mode
        uo = self._payload_offsets(raw, frame0, nframe)
        kernels.mark4_state_counts(raw, uo, nframe, nchan, fanout, ft, counts,
                                   set_origin=origin, sets_per_bin=per_bin)

    def _payload_offsets(self, raw, frame0, nframe):
        """Header scan of a chunk: payload offset of every frame (< 0:
        invalid)."""
        h0 = self.header0
        # with verify, the time code of track 0 must advance by one frame per
        # frame: the scan kernel compares the BCD words with those the writer
        # would generate for the frame's position
        check = None
        if self._index is not None:
            # irregular stream: frames sit where the index says
            rel = self._chunk_layout(frame0, nframe)[4][:, 0]
            _, uo = kernels.mark4_scan(
                raw, nframe, h0.ntrack, frame_offset=torch.from_numpy(
                    np.ascontiguousarray(rel)).to(raw.device),
                want_words=False)
        else:
            if self.verify:
                if self._tick is None:
                    self._tick = _tick_grid(h0, self._frame_rate)
                check = (frame0,) + self._tick
            _, uo = kernels.mark4_scan(
                raw, nframe, h0.ntrack, check=check,
                bad=self._bad_counter(raw.device) if self.verify else None,
                want_words=False)
        return uo

    def _build_index(self):
        """Frame table of an irregular stream, built on the GPU: every place
        where all tracks carry the 32-step all-ones sync word at steps 64..95
        (baseband/mark4/header.py:125-131), with another one a frame later, is
        placed by the BCD time code of track 0 (cf.
        VDIFStreamReader._build_index)."""
        h0 = self.header0
        wordbytes = h0.ntrack // 8
        size = self.fh_raw.seek(0, 2)
        self.fh_raw.seek(0)
        nphys = (size - self._file_offset0) // h0.frame_nbytes
        mjd0, tick0, tick_step = _tick_grid(h0, self._frame_rate)
        nset_max = 2 * nphys + int(round(self._frame_rate)) + 2
        import datetime
        date = datetime.date(1858, 11, 17) + datetime.timedelta(mjd0)
        yday0 = date.timetuple().tm_yday

        def ndays(year):
            return 366 if (year % 4 == 0 and year % 100 != 0) \
                or year % 400 == 0 else 365

        def index_chunk(raw, base, locations, count, table, stats):
            kernels.mark4_index(raw, base, locations, count, h0.ntrack, 0,
                                date.year, yday0, ndays(date.year),
                                ndays(date.year - 1), tick0, tick_step,
                                nset_max, table, stats)

        pattern = np.full(32 * wordbytes, 0xff, np.uint8)
        table, stats = self._build_index_on_device(
            pattern, pattern, h0.frame_nbytes, index_chunk, 1, nset_max,
            pattern_offset=64 * wordbytes)
        self._set_index_table(table, h0.frame_nbytes)

    def read(self, count=None, out=None, **kwargs):
        offset = self.offset
        result = super().read(count, out, **kwargs)
        if self._index is None and self._new_inconsistencies():
            if not self.verify:
                raise OSError('Mark 4 stream is not a regular sequence of '
                              'frames and verify is off.')
            import warnings
            warnings.warn('Mark 4 stream has missing or out-of-order '
                          'frames; indexing all headers and filling the '
                          'gaps with fill_value.')
            self._build_index()
            self.offset = offset
            # "everything" means everything the index knows of
            return super().read(None if count is None and out is None
                                else result.shape[0], out, **kwargs)
        return result


def _tick_grid(h0, frame_rate):
    """(mjd0, tick0, tick_step): the frame times as integer ticks of 0.25 ms
    after 00:00 of MJD mjd0 (Mark 4 times sit on a 1.25 ms grid)."""
    from fractions import Fraction
    t0 = h0.time
    step = Fraction(4000) / Fraction(frame_rate).limit_denominator(10**9)
    start = t0.sec * 4000
    if step.denominator != 1 or Fraction(start).denominator != 1:
        raise ValueError('Mark 4 frame times must lie on the 0.25 ms grid.')
    return int(t0.mjd), int(start), int(step)


def _time_fields(h0, frame_rate, index0, nframe):
    """BCD time-code fields (unit year, day of year, hour, minute, second,
    millisecond) for frames index0.. relative to ``h0``, vectorised.  Mark 4
    times sit on a 1.25 ms grid, so everything is done in integer ticks of
    0.25 ms."""
    from fractions import Fraction
    t0 = h0.time
    step = Fraction(4000) / Fraction(frame_rate).limit_denominator(10**9)
    start = t0.sec * 4000
    if step.denominator != 1 or Fraction(start).denominator != 1:
        raise ValueError('Mark 4 frame times must lie on the 0.25 ms grid.')
    ticks = int(start) + int(step) * np.arange(index0, index0 + nframe,
                                               dtype=np.int64)
    day, tick = np.divmod(ticks, 86400 * 4000)
    date = (np.datetime64('1858-11-17') + (t0.mjd + day).astype(
        'timedelta64[D]'))
    year = date.astype('datetime64[Y]')
    yday = (date - year.astype('datetime64[D]')).astype(np.int64) + 1
    year = year.astype(np.int64) + 1970
    sec, quarter_ms = np.divmod(tick, 4000)
    return np.stack([year % 10, yday, sec // 3600, sec // 60 % 60, sec % 60,
                     quarter_ms // 4], 1)


def _time_words(h0, frame_rate, index0, nframe):
    """Header words 3 and 4 (CRC bits zero) as int32, shape (nframe, 2)."""
    f = _time_fields(h0, frame_rate, index0, nframe)
    w3 = ((bcd_encode(f[:, 0]) << 28) | (bcd_encode(f[:, 1]) << 16)
          | (bcd_encode(f[:, 2]) << 8) | bcd_encode(f[:, 3]))
    w4 = (bcd_encode(f[:, 4]) << 24) | (bcd_encode(f[:, 5]) << 12)
    return np.stack([w3, w4], 1).astype(np.uint32).view(np.int32)


class Mark4StreamWriter(StreamWriterBase):
    """Mark 4 stream writer (GPU encode).  Every frame gets ``header0`` with
    its time code advanced and the CRC-12 of each track recomputed."""
    _sample_shape_maker = Mark4Payload._sample_shape_maker

    def __init__(self, fh_raw, header0=None, sample_rate=None, squeeze=True,
                 device=None):
        fh_raw = Mark4FileWriter(fh_raw)
        super().__init__(fh_raw, header0, sample_rate=sample_rate,
                         squeeze=squeeze, device=device)
        coder = Mark4Payload(np.zeros(
            header0.payload_nbytes // header0.stream_dtype.itemsize,
            header0.stream_dtype), header0)._coder
        try:
            self._mode = codecs._M4_MODES[coder]
        except KeyError:
            raise ValueError('Mark4Payload cannot encode data with {} bits'
                             .format(coder))

    def _encode_frames(self, flat, index0, nframe, valid):
        h0 = self.header0
        dev = flat.device
        nchan, fanout, ft = self._mode
        ntrack = h0.ntrack
        # headers: same words for all frames, time code per frame
        tw = _time_words(h0, self._frame_rate, index0, nframe).view(np.uint32)
        words = np.broadcast_to(h0.words, (nframe, 5, ntrack)).copy()
        words[:, 3, :] = tw[:, 0, None]
        words[:, 4, :] = tw[:, 1, None]
        if not valid.all():
            words[~valid, 1, :] |= np.uint32(1 << 12)   # communication_error
        stream = words2stream(words)                     # (nframe, 160)
        crc = crc_of_bits(np.ascontiguousarray(stream[:, :-12].T), CRC12)
        stream[:, -12:] = crc.T
        frames, uo = kernels.frames_assemble(
            torch.from_numpy(stream.view(np.uint8).reshape(
                nframe, h0.nbytes)).to(dev), h0.frame_nbytes)
        kernels.mark4_encode(flat, frames.view(-1), uo, nframe, nchan, fanout,
                             ft)
        return frames.view(-1)


open = make_opener('mark4', {'rb': Mark4FileReader, 'wb': Mark4FileWriter,
                             'rs': Mark4StreamReader,
                             'ws': Mark4StreamWriter},
                   header_class=Mark4Header,
                   non_header_keys={'sample_rate'},
                   doc="""Open Mark 4 file(s) for reading or writing.

Reader options: ``ntrack`` (determined from the data if omitted), ``decade``
or ``ref_time`` (required), ``sample_rate``, ``squeeze``, ``subset``,
``fill_value``, ``verify``, ``device``.  Writer: ``header0`` or header
keywords (``ntrack``, ``time``, ``bps``, ``fanout`` or ``samples_per_frame``,
``nsb`` ...), ``sample_rate``, ``squeeze``, ``device``.
""")
