"""DADA file and stream readers/writers (API of baseband/dada/base.py).

A DADA file is one (possibly very large) frame, or a sequence of equal frames
the last of which may be cut short (dada/base.py:277-332).  Since samples are
stored time-major, the stream reader does not batch by frames but cuts the
payloads into pieces of ``chunk_nbytes`` on sample boundaries; each piece is
one launch of the int8 kernel.
"""
import numpy as np

from ..base.opener import make_opener
from ..base.stream import (StreamReaderBase, StreamWriterBase,
                           read_file_into)
from ..base.utils import lcm
from ..vdif.base import _FileBase
from .frame import DADAFrame
from .header import DADAHeader
from .payload import DADAPayload, decode_device, HEAP

__all__ = ['DADAFileReader', 'DADAFileWriter', 'DADAStreamReader',
           'DADAStreamWriter', 'open']


class DADAFileReader(_FileBase):
    def read_header(self):
        return DADAHeader.fromfile(self.fh_raw)

    def read_frame(self, memmap=True, verify=True):
        return DADAFrame.fromfile(self.fh_raw, memmap=memmap, verify=verify)

    def get_frame_rate(self):
        with self.temporary_offset(0):
            header = self.read_header()
        return header.sample_rate / header.samples_per_frame


class DADAFileWriter(_FileBase):
    def write_frame(self, data, header=None, **kwargs):
        if not isinstance(data, DADAFrame):
            data = DADAFrame.fromdata(data, header, **kwargs)
        return data.tofile(self.fh_raw)

    def memmap_frame(self, header=None, **kwargs):
        """Write the header now and map the payload, so that the frame can
        be filled in pieces by assigning to slices of it
        (dada/base.py:185-208)."""
        if header is None:
            header = DADAHeader.fromvalues(**kwargs)
        header.tofile(self.fh_raw)
        payload = DADAPayload.fromfile(self.fh_raw, memmap=True,
                                       header=header)
        return DADAFrame(header, payload)


class _DADAStreamBase:
    _sample_shape_maker = DADAPayload._sample_shape_maker

    def _get_index(self, header):
        return int(round((header['OBS_OFFSET'] - self.header0['OBS_OFFSET'])
                         / self.header0.payload_nbytes))

    def _set_index(self, header, index):
        header.update(obs_offset=self.header0['OBS_OFFSET']
                      + index * self.header0.payload_nbytes)


class DADAStreamReader(_DADAStreamBase, StreamReaderBase):
    """DADA stream reader (GPU decode)."""

    def __init__(self, fh_raw, squeeze=True, subset=(), verify=True,
                 device=None, chunk_nbytes=None, dtype=None):
        fh_raw = DADAFileReader(fh_raw)
        header0 = fh_raw.read_header()
        size = fh_raw.seek(0, 2)
        nframe, partial = divmod(size, header0.frame_nbytes)
        self._last_nbytes = header0.payload_nbytes
        if partial > header0.nbytes:
            # truncated last frame: whole words and whole samples only
            sample_nbytes = (header0.bps * (2 if header0.complex_data else 1)
                             * header0['NPOL'] * header0['NCHAN']) // 8
            block = lcm(4, sample_nbytes)
            self._last_nbytes = (partial - header0.nbytes) // block * block
            nframe += 1
        elif nframe == 0:
            raise EOFError('file (of {0} bytes) appears to end without any '
                           'payload.'.format(partial))
        self._nframe = nframe
        spf = header0.samples_per_frame
        if nframe == 1 and self._last_nbytes != header0.payload_nbytes:
            spf = self._last_nbytes * 8 // header0._bits_per_sample
        self._mkbf = header0.get('INSTRUMENT') == 'MKBF'
        super().__init__(fh_raw, header0, squeeze=squeeze, subset=subset,
                         verify=verify, samples_per_frame=spf, device=device,
                         chunk_nbytes=chunk_nbytes, dtype=dtype)
        self._sample_nbytes = header0._bits_per_sample // 8
        self._last_nsample = self._last_nbytes // self._sample_nbytes

    @property
    def _nsample(self):
        return (self._nframe - 1) * self._samples_per_frame \
            + self._last_nsample

    @property
    def _frame_nbytes(self):
        return self.header0.frame_nbytes

    def _chunks(self, start, count):
        """Pieces never span frames: (frame, 1, local start, n, row)."""
        if count == 0:
            return
        spf = self._samples_per_frame
        step = max(1, self._chunk_nbytes // self._sample_nbytes)
        if self._mkbf:
            step = max(HEAP, step // HEAP * HEAP)
        pos, row = start, 0
        while row < count:
            frame, local = divmod(pos, spf)
            in_frame = (self._last_nsample if frame == self._nframe - 1
                        else spf)
            n = min(count - row, in_frame - local, step - local % step
                    if self._mkbf else step)
            yield frame, 1, local, n, row
            pos += n
            row += n

    def _piece(self, local, n):
        """Byte range (relative to the payload) needed for samples
        [local, local + n), 4-byte aligned, and the sample it starts at."""
        unit = HEAP if self._mkbf else 1
        s0 = local // unit * unit
        b0 = s0 * self._sample_nbytes
        shift = b0 % 4
        if shift:          # align start down to a word: whole samples only
            per = lcm(4, self._sample_nbytes) // self._sample_nbytes
            s0 = s0 // per * per
            b0 = s0 * self._sample_nbytes
        s1 = -(-(local + n) // unit) * unit
        b1 = -(-(s1 * self._sample_nbytes) // 4) * 4
        return s0, b0, b1

    def _chunk_nbytes_of(self, frame0, nframe, sample_start, nsample):
        s0, b0, b1 = self._piece(sample_start, nsample)
        limit = (self._last_nbytes if frame0 == self._nframe - 1
                 else self.header0.payload_nbytes)
        return min(b1, limit) - b0

    def _read_raw(self, frame0, nframe, pinned, sample_start=0, nsample=0):
        s0, b0, b1 = self._piece(sample_start, nsample)
        view = pinned.numpy()
        if read_file_into(self.fh_raw, frame0 * self.header0.frame_nbytes
                          + self.header0.nbytes + b0, view) != view.size:
            raise EOFError('could not read payload bytes of frame {}.'
                           .format(frame0))

    def _decode_chunk(self, raw, frame0, nframe, sample_start, nsample, out):
        h0 = self.header0
        if h0.bps != 8:
            raise KeyError(h0.bps)
        s0, b0, b1 = self._piece(sample_start, nsample)
        decode_device(raw, 0, raw.numel(), h0['NPOL'], h0['NCHAN'],
                      h0.complex_data, self._mkbf, sample_start - s0,
                      nsample, out)

    # -- packed consumers (tasks.moments) -----------------------------------
    def _for_each_packed_chunk(self, frame0, nframe, fn):
        """The base loop works on whole frames; DADA frames can be far larger
        than a chunk, so the pieces of `_chunks` (never spanning frames) go
        through the same three-stage pipeline and ``fn`` sees each as part of
        its frame (``fn(raw, frame, 1)``, the piece being the one unit)."""
        if self._mkbf:
            raise NotImplementedError('packed consumers do not know the MKBF '
                                      'heap layout')
        from ..base.stream import DEVICE_READ_STAGES
        dev = self.device
        stages, ss = self._pipeline(dev)
        spf = self._samples_per_frame
        word = lcm(4, self._sample_nbytes)
        chunks = list(self._chunks(frame0 * spf, nframe * spf))
        for f0, nf, s0, ns, _ in chunks:
            if (s0 * self._sample_nbytes) % 4 or (ns * self._sample_nbytes) % 4:
                raise ValueError('chunk_nbytes must hold whole words of whole '
                                 'samples ({} bytes) for a packed consumer'
                                 .format(word))
        ss.after_caller(1)

        def begin(k):
            f0, nf, s0, ns, _ = chunks[k]
            st = stages[k % DEVICE_READ_STAGES]
            if st.done is not None:
                st.done.synchronize()
            pin, _ = st.buffers(self._chunk_nbytes_of(f0, nf, s0, ns), 0, dev,
                                False)
            return self._read_raw_begin(f0, nf, pin, s0, ns)

        ahead = begin(0) if chunks else None
        for k, (f0, nf, s0, ns, _) in enumerate(chunks):
            st = stages[k % DEVICE_READ_STAGES]
            raw = st.raw[:self._chunk_nbytes_of(f0, nf, s0, ns)]
            pin = ahead.wait()
            ahead = begin(k + 1) if k + 1 < len(chunks) else None
            try:
                with ss.use(0):
                    ss.wait_event(0, st.free)
                    self._upload(raw, pin, f0, nf)
                    st.done = ss.event(0)
                with ss.use(1):
                    ss.wait_event(1, st.done)
                    fn(raw[:ns * self._sample_nbytes], f0, 1)
                    st.free = ss.event(1)
            except BaseException:
                if ahead is not None:
                    ahead.wait()
                raise
        ss.caller_after(1)

    def _packed_units(self, raw, frame0, nframe):
        """``raw`` is one piece of one frame's payload: a single unit."""
        import torch
        h0 = self.header0
        if h0.bps != 8:
            raise KeyError(h0.bps)
        ib = 2 if h0.complex_data else 1
        uo = torch.zeros(1, dtype=torch.int64).to(raw.device)
        return uo, 1, raw.numel(), 8, h0['NPOL'] * h0['NCHAN'] * ib

    def _moments_view(self, m):
        """(nbin, 1, npol * nchan * parts, 3) -> (nbin, npol, nchan, parts)."""
        h0 = self.header0
        ib = 2 if h0.complex_data else 1
        m = m.reshape(m.shape[0], h0['NPOL'], h0['NCHAN'], ib, 3)
        return m if ib == 2 else m[..., 0, :]

    @property
    def stop_time(self):
        return self.start_time + self._offset_seconds(self._nsample)


class DADAStreamWriter(_DADAStreamBase, StreamWriterBase):
    """DADA stream writer (GPU encode): every frame is ``header0`` with
    ``OBS_OFFSET`` advanced, followed by the encoded payload."""

    def __init__(self, fh_raw, header0, squeeze=True, device=None):
        fh_raw = DADAFileWriter(fh_raw)
        super().__init__(fh_raw, header0, squeeze=squeeze, device=device)

    def _encode_frames(self, flat, index0, nframe, valid):
        import io
        import torch
        from .. import kernels
        h0 = self.header0
        dev = flat.device
        if h0.bps != 8:
            raise ValueError('DADAPayload cannot encode data with {} bits'
                             .format(h0.bps))
        texts = []
        for i in range(nframe):
            header = h0.copy()
            header.mutable = True
            self._set_index(header, index0 + i)
            with io.BytesIO() as s:
                header.tofile(s)
                texts.append(np.frombuffer(s.getvalue(), np.uint8))
        headers = torch.from_numpy(np.stack(texts)).to(dev)
        ib = 2 if h0.complex_data else 1
        nelem = h0['NPOL'] * h0['NCHAN'] * ib
        if h0.get('INSTRUMENT') == 'MKBF':
            heap_nbytes = nelem * HEAP
            per = h0.payload_nbytes // heap_nbytes
            frames, uo = kernels.frames_assemble(
                headers, h0.frame_nbytes, units_per_frame=per,
                unit_stride=heap_nbytes)
            kernels.encode_int8_transposed(flat, frames.view(-1), uo,
                                           nframe * per,
                                           h0['NPOL'] * h0['NCHAN'], HEAP, ib)
        else:
            frames, uo = kernels.frames_assemble(headers, h0.frame_nbytes)
            kernels.encode_bitfield(flat, frames.view(-1), uo, nframe, 1,
                                    h0.payload_nbytes, 8, nelem,
                                    kernels.QUANT_SINT)
        return frames.view(-1)


open = make_opener('dada', {'rb': DADAFileReader, 'wb': DADAFileWriter,
                            'rs': DADAStreamReader, 'ws': DADAStreamWriter},
                   header_class=DADAHeader,
                   doc="""Open DADA file(s) for reading or writing.

Reader options: ``squeeze``, ``subset``, ``verify``, ``device``.  Writer:
``header0`` or header keywords (``time``, ``sample_rate``,
``samples_per_frame``, ``sample_shape``, ``bps``, ``complex_data`` ...),
``squeeze``, ``device``.
""")
