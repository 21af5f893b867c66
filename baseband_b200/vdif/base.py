"""VDIF file and stream readers/writers.

API of baseband/vdif/base.py (file reader :70-314, stream reader :401-534,
stream writer :758-807, ``open`` :810-884).  The stream reader decodes whole
ranges of frame sets per kernel launch: ``bb_vdif_scan`` parses every header
of a chunk on the GPU (invalid flag, thread id -> output slot, payload
offset) and ``bb_decode_bitfield`` unpacks all payloads straight into
``(nsample, nthread, nchan)``.
"""
import numpy as np
import torch

from .. import kernels
from ..base.opener import make_opener
from ..base.stream import StreamReaderBase, StreamWriterBase, as_hertz
from .frame import VDIFFrame, VDIFFrameSet
from .header import VDIFHeader
from .payload import VDIFPayload

__all__ = ['VDIFFileReader', 'VDIFFileWriter', 'VDIFStreamReader',
           'VDIFStreamWriter', 'open']


class _FileBase:
    def __init__(self, fh_raw):
        self.fh_raw = fh_raw

    def __getattr__(self, attr):
        if attr == 'fh_raw':
            raise AttributeError(attr)
        return getattr(self.fh_raw, attr)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.fh_raw.close()

    def temporary_offset(self, offset=None, whence=0):
        return _TemporaryOffset(self.fh_raw, offset, whence)

    # sync search around the file pointer (base/base.py:181-376)
    def locate_frames(self, pattern=None, **kwargs):
        """Positions of frames near the current one, nearest first; see
        `baseband_b200.base.locate.locate_frames`.  Without ``pattern`` the
        format's own invariant header bits are used."""
        from ..base import locate
        if pattern is None:
            pattern, extra = self._default_pattern()
            for key, value in extra.items():
                kwargs.setdefault(key, value)
        return locate.locate_frames(self.fh_raw, pattern, **kwargs)

    def find_header(self, *args, **kwargs):
        """Nearest readable header; the file pointer is left at its start."""
        from ..base import locate
        return locate.find_header(self, *args, **kwargs)

    def _default_pattern(self):
        raise TypeError('a pattern (or a header) is needed to locate {} '
                        'frames.'.format(type(self).__name__))


class _TemporaryOffset:
    def __init__(self, fh, offset, whence):
        self.fh, self.offset, self.whence = fh, offset, whence

    def __enter__(self):
        self.saved = self.fh.tell()
        if self.offset is not None:
            self.fh.seek(self.offset, self.whence)
        return self.fh

    def __exit__(self, *exc):
        self.fh.seek(self.saved)


class VDIFFileReader(_FileBase):
    """Binary-level reader: headers, frames, frame sets."""

    def read_header(self, edv=None, verify=True):
        return VDIFHeader.fromfile(self.fh_raw, edv=edv, verify=verify)

    def read_frame(self, edv=None, verify=True):
        return VDIFFrame.fromfile(self.fh_raw, edv=edv, verify=verify)

    def read_frameset(self, thread_ids=None, edv=None, verify=True):
        return VDIFFrameSet.fromfile(self.fh_raw, thread_ids, edv=edv,
                                     verify=verify)

    def get_thread_ids(self, check=2):
        """Sorted thread ids found in the first frame sets: scan until the
        set of ids has not grown for ``check`` frame numbers
        (vdif/base.py:172-215)."""
        with self.temporary_offset():
            header = header0 = self.read_header()
            ids = set()
            remaining = 1
            try:
                while remaining > 0:
                    frame_nr, before = header['frame_nr'], len(ids)
                    while header['frame_nr'] == frame_nr:
                        ids.add(header['thread_id'])
                        self.fh_raw.seek(header.payload_nbytes, 1)
                        header = self.read_header(edv=header0.edv)
                    remaining = check if len(ids) > before else remaining - 1
            except EOFError:
                pass          # short file: every frame has been looked at
        return sorted(ids)

    def get_frame_rate(self):
        """Frames per second: highest frame number within a second, plus one
        (base/base.py:371-406); falls back on the header's sample rate."""
        with self.temporary_offset(0):
            try:
                header = header0 = self.read_header()
                frame_nr0 = header['frame_nr']
                while header['frame_nr'] == frame_nr0:
                    self.fh_raw.seek(header.payload_nbytes, 1)
                    header = self.read_header()
                highest = frame_nr0
                while header['frame_nr'] > 0:
                    highest = max(highest, header['frame_nr'])
                    self.fh_raw.seek(header.payload_nbytes, 1)
                    header = self.read_header()
                return float(highest + 1)
            except Exception as exc:
                rate = getattr(header0, 'sample_rate', None) \
                    if 'header0' in locals() else None
                if rate:
                    return float(round(rate / header0.samples_per_frame))
                raise exc


class VDIFFileWriter(_FileBase):
    def write_frame(self, data, header=None, **kwargs):
        if not isinstance(data, VDIFFrame):
            data = VDIFFrame.fromdata(data, header, **kwargs)
        return data.tofile(self.fh_raw)

    def write_frameset(self, data, header=None, **kwargs):
        if not isinstance(data, VDIFFrameSet):
            data = VDIFFrameSet.fromdata(data, header, **kwargs)
        return data.tofile(self.fh_raw)


class _VDIFStreamBase:
    def _get_index(self, header):
        # vdif/base.py:386-390
        h0 = self.header0
        return int(round((header['seconds'] - h0['seconds'])
                         * self._frame_rate
                         + header['frame_nr'] - h0['frame_nr']))

    def _get_time(self, header):
        return header.get_time(frame_rate=self._frame_rate)

    def _set_time(self, header, time):
        header.set_time(time, frame_rate=self._frame_rate)


class VDIFStreamReader(_VDIFStreamBase, StreamReaderBase):
    """VDIF stream reader (GPU decode).

    Parameters as the reference (``sample_rate``, ``squeeze``, ``subset``,
    ``fill_value``, ``verify``) plus ``device`` and ``chunk_nbytes``.
    """
    def __init__(self, fh_raw, sample_rate=None, squeeze=True, subset=(),
                 fill_value=0., verify='fix', device=None,
                 chunk_nbytes=None, dtype=None):
        fh_raw = VDIFFileReader(fh_raw)
        header0 = fh_raw.read_header()
        fh_raw.seek(0)
        thread_ids = fh_raw.get_thread_ids()
        self._file_thread_ids = thread_ids
        nthread = len(thread_ids)
        sample_rate = as_hertz(sample_rate)
        if sample_rate is None:
            sample_rate = getattr(header0, 'sample_rate', None) or None
        if sample_rate is None:
            sample_rate = fh_raw.get_frame_rate() * header0.samples_per_frame
        self._set_nbytes = header0.frame_nbytes * nthread
        size = fh_raw.seek(0, 2)
        fh_raw.seek(0)
        self._nframe = size // self._set_nbytes
        super().__init__(
            fh_raw, header0, sample_rate=sample_rate,
            sample_shape=(nthread, header0.nchan), squeeze=squeeze,
            subset=subset, fill_value=fill_value, verify=verify,
            device=device, chunk_nbytes=chunk_nbytes, dtype=dtype)
        # Split the subset into thread selection (done by the scan kernel's
        # slot table, so unwanted threads are never decoded) and the rest,
        # applied after decoding (vdif/base.py:464-490).
        if self._subset and (nthread > 1 or not self._squeeze):
            picked = np.array(thread_ids)[self._subset[0]]
            self._thread_ids = np.atleast_1d(picked.squeeze()).tolist()
            if picked.shape == ():
                first = () if self._squeeze else (0,)
            elif len(self._thread_ids) == 1 and self._squeeze:
                first = (np.newaxis,)
            else:
                first = (slice(None),)
            self._post_subset = first + self._subset[1:]
        else:
            self._post_subset = self._subset
            self._thread_ids = list(thread_ids)
        # A selection may name a thread more than once (subset [0, -1] on a
        # one-thread file): each thread is decoded once and duplicates are
        # expanded by a gather on the decoded samples.
        self._decode_ids = list(dict.fromkeys(self._thread_ids))
        self._thread_expand = None
        if len(self._decode_ids) != len(self._thread_ids):
            self._thread_expand = [self._decode_ids.index(t)
                                   for t in self._thread_ids]
        slots = np.full(1024, -1, np.int32)
        for slot, tid in enumerate(self._decode_ids):
            slots[tid] = slot
        self._slots_host = slots
        self._slots_dev = None
        self._index = None
        if self.verify:
            # A partial frame set at the end of the file, or a last frame
            # whose time does not match its position, means frames were lost
            # somewhere: index all headers right away.
            lossy = size % self._set_nbytes != 0
            if not lossy and size >= header0.frame_nbytes:
                # last frame of the thread the first header belongs to (some
                # recorders time-stamp only part of the threads correctly,
                # cf. vdif/base.py:492-517)
                try:
                    for back in range(1, nthread + 1):
                        fh_raw.seek(size - back * header0.frame_nbytes)
                        last = fh_raw.read_header(edv=header0.edv)
                        if last['thread_id'] == header0['thread_id']:
                            lossy = (self._get_index(last)
                                     != self._nframe - 1)
                            break
                    else:
                        lossy = True
                except Exception:
                    lossy = True
                fh_raw.seek(0)
            if lossy:
                self._build_index()
        fn = (VDIFPayload(np.zeros(header0.payload_nbytes // 4, '<u4'),
                          header0)._decoders[header0.bps])
        self._codec = (fn.codec, fn.levels)

    _sample_shape_maker = None

    @property
    def _unsliced_shape(self):
        from collections import namedtuple
        return namedtuple('SampleShape', 'nthread, nchan')(
            *self._sample_shape)

    @property
    def _frame_nbytes(self):
        return self._set_nbytes

    # decoded layout: selected threads only
    @property
    def _floats_per_sample(self):
        return (len(self._decode_ids) * self._sample_shape[1]
                * (2 if self._complex_data else 1))

    def _finish(self, flat, nsample):
        nthread, nchan = len(self._decode_ids), self._sample_shape[1]
        n = nsample * self._floats_per_sample
        if self._complex_data:
            data = self._complex_view(flat[:n].view(nsample, nthread,
                                                    nchan, 2))
        else:
            data = flat[:n].view(nsample, nthread, nchan)
        if self._thread_expand is not None:
            data = data[:, torch.as_tensor(self._thread_expand,
                                           device=data.device)]
        if self._squeeze:
            data = data.reshape((nsample,) + tuple(
                d for d in data.shape[1:] if d > 1))
        if self._post_subset:
            from ..base.stream import _torch_index
            data = data[(slice(None),) + _torch_index(self._post_subset,
                                                      data.device)]
        return data

    def _decode_chunk(self, raw, frame0, nframe, sample_start, nsample, out):
        uo, nthread, payload_nbytes, bps, nelem = self._packed_units(
            raw, frame0, nframe)
        kernels.decode_bitfield(
            raw, uo, nframe, nthread, payload_nbytes, bps, nelem,
            self._complex_data, self._codec[0], self._codec[1],
            self._fill_value, sample_start, nsample, out)

    def _packed_units(self, raw, frame0, nframe):
        h0 = self.header0
        dev = raw.device
        nelem = self._sample_shape[1] * (2 if self._complex_data else 1)
        if self._index is not None:
            # irregular stream: unit table from the frame index (where each
            # frame of the chunk was put on the device: `_chunk_layout`)
            rel = self._chunk_layout(frame0, nframe)[4]
            uo = np.where(rel >= 0, rel + h0.nbytes, -1)
            uo = torch.from_numpy(np.ascontiguousarray(uo.reshape(-1))).to(dev)
        else:
            if self._slots_dev is None or self._slots_dev.device != dev:
                self._slots_dev = torch.from_numpy(self._slots_host).to(dev)
            nthread_file = len(self._file_thread_ids)
            # with verify, every set must also carry the frame index its
            # position implies: checked inside the scan kernel
            check = ((frame0, h0['seconds'], h0['frame_nr'],
                      int(round(self._frame_rate))) if self.verify else None)
            _, uo, _ = kernels.vdif_scan(
                raw, nframe * nthread_file, h0.frame_nbytes, h0.nbytes,
                nthread_file, self._slots_dev, len(self._decode_ids),
                check=check, bad=self._bad_counter(dev), want_fields=False)
        return uo, len(self._decode_ids), h0.payload_nbytes, h0.bps, nelem

    # ------------------------------------------- irregular (lossy) streams
    def _build_index(self):
        """Frame table for streams with missing, duplicated or re-ordered
        frames, or with bytes lost or inserted between frames (the losses of
        network recorders; the reference repairs these one frame at a time in
        ``_bad_frame``, vdif/base.py:536-755, on top of `locate_frames`,
        base/base.py:181-335).  Built on the GPU (`_build_index_on_device`):
        every header that matches the stream's invariant header bits
        (vdif/header.py:109-115) and is followed by another such header one
        frame on is assigned to (set index, thread slot) from its seconds /
        frame_nr / thread_id; the first such frame in the file wins, frames
        flagged invalid count as missing.  Installs an int64 table
        ``(nset, nthread)`` of frame byte offsets, -1 where there is none."""
        h0 = self.header0
        dev = self.device
        size = self.fh_raw.seek(0, 2)
        self.fh_raw.seek(0)
        nphys = size // h0.frame_nbytes
        fps = int(round(self._frame_rate))
        nthread_file = max(1, len(self._file_thread_ids))
        nslot = len(self._decode_ids)
        nset_max = 2 * (nphys // nthread_file) + fps + 2
        pattern, mask = h0.invariant_pattern()
        if self._slots_dev is None or self._slots_dev.device != dev:
            self._slots_dev = torch.from_numpy(self._slots_host).to(dev)

        def index_chunk(raw, base, locations, count, table, stats):
            kernels.vdif_index(raw, base, locations, count, self._slots_dev,
                               nslot, h0['seconds'], h0['frame_nr'], fps,
                               nset_max, table, stats,
                               thread0=h0['thread_id'])

        table, stats = self._build_index_on_device(
            pattern, mask, h0.frame_nbytes, index_chunk, nslot, nset_max)
        # the stream ends with the last good frame of the first header's
        # thread, as in the reference (vdif/base.py:493-519)
        table = table[:int(stats[3]) + 1]
        # A header not followed by another one is normally the frame before
        # a break (its payload may be short).  The last such frame of the
        # stream is different: what follows it is beyond the end of the
        # stream, and the reference, which stops at its last good header,
        # reads it as it stands.
        last = int(table.max()) if table.size else -1
        for loc in self._index_loose:
            if loc <= last or loc + h0.frame_nbytes > size:
                continue
            self.fh_raw.seek(int(loc))
            try:
                header = self.fh_raw.read_header(edv=h0.edv)
            except Exception:
                continue
            finally:
                self.fh_raw.seek(0)
            index = ((header['seconds'] - h0['seconds']) * fps
                     + header['frame_nr'] - h0['frame_nr'])
            slot = int(self._slots_host[header['thread_id']])
            if (0 <= index < table.shape[0] and 0 <= slot < nslot
                    and table[index, slot] < 0
                    and not header['invalid_data']):
                table[index, slot] = loc
        self._index_stats = {'frames_outside_table': int(stats[1])}
        self._set_index_table(table, h0.frame_nbytes)

    def read(self, count=None, out=None, **kwargs):
        offset = self.offset
        result = super().read(count, out, **kwargs)
        nbad = self._new_inconsistencies() if self._index is None else 0
        if nbad:
            if not self.verify:
                raise OSError(
                    'VDIF stream is not a regular sequence of complete '
                    'frame sets ({} inconsistent frames) and verify is '
                    'off.'.format(nbad))
            import warnings
            warnings.warn('VDIF stream has missing or out-of-order '
                          'frames; indexing all headers and filling the '
                          'gaps with fill_value.')
            self._build_index()
            self.offset = offset
            # "everything" means everything the index knows of
            n = None if count is None and out is None else result.shape[0]
            return super().read(n, out if out is not None else None, **kwargs)
        return result


class VDIFStreamWriter(_VDIFStreamBase, StreamWriterBase):
    """VDIF stream writer (GPU encode).

    ``header0`` gives the first header; ``nthread`` the number of threads.
    """

    def __init__(self, fh_raw, header0=None, sample_rate=None, nthread=1,
                 squeeze=True, device=None):
        fh_raw = VDIFFileWriter(fh_raw)
        header_rate = getattr(header0, 'sample_rate', None) or None
        sample_rate = as_hertz(sample_rate)
        if sample_rate is None:
            if header_rate is None:
                raise ValueError('the sample rate must be passed either '
                                 'explicitly, or through the header if it '
                                 'can be stored there.')
            sample_rate = header_rate
        elif header_rate is not None:
            assert sample_rate == header_rate, (
                'sample_rate on header inconsistent with that passed in.')
        super().__init__(fh_raw, header0, sample_rate=sample_rate,
                         sample_shape=(nthread, header0.nchan),
                         squeeze=squeeze, device=device)
        self._nthread = nthread
        self._quantiser = (kernels.QUANT_MARK5B if header0.edv == 0xab
                           else kernels.QUANT_OFFSET_BINARY)

    @property
    def _unsliced_shape(self):
        from collections import namedtuple
        return namedtuple('SampleShape', 'nthread, nchan')(
            *self._sample_shape)

    def _encode_frames(self, flat, index0, nframe, valid):
        h0 = self.header0
        dev = flat.device
        nthread, nw = self._nthread, h0.nbytes // 4
        fps = int(round(self._frame_rate))
        # headers for every (set, thread): vdif/base.py:392-398
        words = np.empty((nframe, nthread, nw), np.uint32)
        words[:] = np.array([int(w) for w in h0.words], np.uint32)
        index = np.arange(index0, index0 + nframe, dtype=np.int64)
        dt, frame_nr = np.divmod(index + h0['frame_nr'], fps)
        seconds = h0['seconds'] + dt
        words[:, :, 0] = ((words[:, :, 0] & np.uint32(0x40000000))
                          | (seconds[:, None].astype(np.uint32)
                             & np.uint32(0x3fffffff))
                          | (np.uint32(0x80000000)
                             * (~valid[:, None]).astype(np.uint32)))
        words[:, :, 1] = ((words[:, :, 1] & np.uint32(0xff000000))
                          | frame_nr[:, None].astype(np.uint32))
        tids = np.arange(nthread, dtype=np.uint32)
        words[:, :, 3] = ((words[:, :, 3] & np.uint32(~(0x3ff << 16)
                                                     & 0xffffffff))
                          | (tids[None, :] << np.uint32(16)))
        n = nframe * nthread
        # headers into place + unit offsets: one launch (bb_frames_assemble)
        frames, uo = kernels.frames_assemble(
            torch.from_numpy(words.reshape(n, nw)
                             .view(np.uint8)).to(dev), h0.frame_nbytes)
        nelem = self._sample_shape[1] * (2 if self._complex_data else 1)
        kernels.encode_bitfield(flat, frames.view(-1), uo, nframe, nthread,
                                h0.payload_nbytes, h0.bps, nelem,
                                self._quantiser)
        return frames.view(-1)


open = make_opener('vdif', {'rb': VDIFFileReader, 'wb': VDIFFileWriter,
                            'rs': VDIFStreamReader, 'ws': VDIFStreamWriter},
                   header_class=VDIFHeader,
                   non_header_keys={'sample_rate', 'nthread'},
                   doc="""Open VDIF file(s) for reading or writing.

Modes 'rb'/'wb' give binary frame-level access; 'rs'/'ws' (default 'rs')
stream samples.  Stream options: ``sample_rate``, ``squeeze``, ``subset``,
``fill_value``, ``verify`` (reading); ``header0`` or header keywords,
``sample_rate``, ``nthread``, ``squeeze`` (writing); and for both ``device``
(CUDA device; reads then return torch tensors that stay on the GPU).
""")
