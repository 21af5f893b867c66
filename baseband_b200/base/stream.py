"""Stream readers and writers: samples in, samples out, frames batched on GPU.

Public surface follows the reference's stream classes
(baseband/base/base.py:409-1342): ``read(count=None, out=None)``, ``seek``,
``tell``, ``shape``, ``sample_shape``, ``dtype``, ``start_time``, ``stop_time``,
``fill_value``, ``squeeze``, ``subset``; ``write(data, valid=True)``,
``close``.  What differs is the execution model.  The reference walks the
file one frame at a time in Python (base/base.py:957-967); here a ``read``
turns the requested sample range into a range of frames, streams their raw
bytes through pinned host buffers to the GPU in large chunks, and per chunk
launches a header-scan kernel (validity, thread slots, payload offsets) and
one decode kernel that writes the final ``(nsample, *sample_shape)`` layout
directly.  Chunks are double buffered over three CUDA streams (H2D, kernels,
D2H) so the PCIe copies overlap the kernels.

Device-output option (north_star): ``open(..., device='cuda:0')`` or passing a
CUDA ``torch.Tensor`` as ``out`` keeps the decoded samples on the GPU.

There is no CPU decode path: without the CUDA library every read raises.
"""
import functools
import mmap
import operator
import os
from collections import namedtuple

import numpy as np
import torch

from .. import device as _device
from ..timeutil import Time, as_time

__all__ = ['StreamBase', 'StreamReaderBase', 'StreamWriterBase',
           'as_hertz', 'DEFAULT_CHUNK_NBYTES']

# Packed bytes per pipeline stage.  A 2-bit stream expands 16x, so 16 MiB of
# frames become 256 MiB of float32 per stage (two stages in flight).  With
# one chunk of read-ahead the per-chunk host work is hidden, and staging
# buffers of this size stay in the host's last-level cache between the copy
# out of the page cache and the DMA read: file ingest peaks at 8-16 MiB
# (profiles/r2_file_chunks.txt: 38-43 GB/s, against 30 at 64 MiB).
DEFAULT_CHUNK_NBYTES = 16 << 20
# stages a device-output read rotates over (see `_pipeline`; 2 or 3)
DEVICE_READ_STAGES = 3

# File -> pinned staging buffer: one readinto() copies out of the page cache on
# a single core (a few GB/s), far below the PCIe link.  Large chunks of plain
# files are therefore copied as several slices on a small thread pool, from a
# read-only mmap of the file: a user-space memcpy out of the mapped page cache
# moves ~15 GB/s per core where the kernel's copy in read()/preadv() manages
# ~6 (profiles/r2_host_copy.txt: 4 threads 43 vs 22 GB/s, 8 threads 66 vs
# 36), which keeps the H2D copy fed with half the cores.  The slices run on the
# library's pool of native threads (bb_host_copy; bb_host_pread where mmap is
# refused): a Python thread pool costs ~50 us per slice, as much as the copy
# of a small chunk.
# (from 2 MiB on: a `chunk_nbytes` of 8 MiB is a little less than 8 MiB of whole
# frames, and fell back to the single readinto -- 7 instead of 40 GB/s)
PARALLEL_READ_MIN_NBYTES = 2 << 20
PARALLEL_READ_MMAP = True
# read(out=<pageable numpy array>) at least this large: staged D2H (see
# StreamReaderBase._read_to_host).
STAGED_HOST_OUT_MIN_NBYTES = 4 << 20
PARALLEL_READ_THREADS = max(1, min(8, len(os.sched_getaffinity(0))
                                   if hasattr(os, 'sched_getaffinity')
                                   else (os.cpu_count() or 1)))
def _plain_file(fh):
    """``(io.FileIO, fd)`` of the plain binary file behind ``fh``, or None:
    anything else with a fileno() (gzip, ...) would hand out the bytes of the
    file underneath it."""
    import io
    import stat
    plain = fh
    while hasattr(plain, 'fh_raw'):
        plain = plain.fh_raw
    raw = plain.raw if isinstance(plain, (io.BufferedReader,
                                          io.BufferedRandom)) else plain
    if not isinstance(raw, io.FileIO):
        return None
    try:
        fd = raw.fileno()
        if not stat.S_ISREG(os.fstat(fd).st_mode):
            return None
    except (OSError, ValueError):
        return None
    return raw, fd


def _parallel_readinto(fh, offset, view):
    """Fill the writable uint8 numpy array ``view`` from absolute byte
    ``offset`` of the plain file behind ``fh``.  Returns the bytes read, or
    None if ``fh`` is not a plain file (the caller falls back to
    ``readinto``)."""
    if PARALLEL_READ_THREADS < 1:
        return None
    plain = _plain_file(fh)
    if plain is None:
        return None
    raw, fd = plain
    import ctypes
    from .._lib import host_io
    lib = host_io()
    n = view.size
    dst = ctypes.c_void_p(view.ctypes.data)
    mapped = _mapped_file(raw, fd, offset + n) if PARALLEL_READ_MMAP else None
    if mapped is not None:
        # user-space memcpy out of the mapped page cache, native threads
        arr = mapped[1]
        n = max(0, min(n, arr.size - offset))
        rc = lib.bb_host_copy(dst, ctypes.c_void_p(arr.ctypes.data + offset),
                              n, PARALLEL_READ_THREADS)
        return n if rc == 0 else None
    nread = ctypes.c_int64(0)
    rc = lib.bb_host_pread(fd, dst, n, offset, PARALLEL_READ_THREADS,
                           ctypes.byref(nread))
    return int(nread.value) if rc == 0 else None


class _Ready:
    """A chunk read that is already complete."""
    def __init__(self, value):
        self.value = value

    def wait(self):
        return self.value


class _PendingCopy:
    """A chunk being copied into pinned staging by the library's thread pool
    (bb_host_copy_begin); `wait` returns the staging tensor."""
    def __init__(self, lib, tensor, nbytes):
        self.lib, self.tensor, self.nbytes = lib, tensor, nbytes

    def wait(self):
        import ctypes
        lib, self.lib = self.lib, None
        if lib is not None:
            moved = ctypes.c_int64(0)
            lib.bb_host_copy_wait(ctypes.byref(moved))
            if moved.value != self.nbytes:
                raise EOFError('could not read a whole chunk of frames.')
        return self.tensor


_file_maps = None


def _mapped_file(raw, fd, need):
    """Read-only mmap of the plain file behind ``raw`` (kept per file object,
    re-made when the file has grown past it) as ``(mmap, uint8 array)``, or
    None if it cannot be mapped."""
    global _file_maps
    if _file_maps is None:
        import weakref
        _file_maps = weakref.WeakKeyDictionary()
    try:
        entry = _file_maps.get(raw)
        if entry is None or entry[1].size < need:
            size = os.fstat(fd).st_size
            if size <= 0:
                return None
            mm = mmap.mmap(fd, size, prot=mmap.PROT_READ)
            entry = (mm, np.frombuffer(mm, np.uint8))
            _file_maps[raw] = entry
        return entry
    except (OSError, ValueError, TypeError):
        return None


def read_file_into(fh, offset, view):
    """Read ``view.size`` bytes at absolute ``offset`` of ``fh`` into the
    uint8 numpy array ``view`` (normally pinned memory) -- in parallel slices
    for large requests on plain files, with ``seek`` + ``readinto``
    otherwise.  Leaves ``fh`` positioned after the bytes read; returns the
    number of bytes read."""
    got = None
    if view.size >= PARALLEL_READ_MIN_NBYTES:
        got = _parallel_readinto(fh, offset, view)
        if got is not None:
            fh.seek(offset + got)
    if got is None:
        fh.seek(offset)
        got = fh.readinto(memoryview(view))
    return got


_TIME_UNITS = {'s': 1.0, 'ms': 1e3, 'us': 1e6, 'ns': 1e9, 'min': 1 / 60.,
               'h': 1 / 3600., 'day': 1 / 86400.}


def as_hertz(rate):
    """A sample rate as float Hz; accepts numbers and astropy Quantities."""
    if rate is None:
        return None
    to_value = getattr(rate, 'to_value', None)
    if to_value is not None:
        return float(to_value('Hz'))
    return float(rate)


def _squeezed(shape):
    """Shape with unit dimensions removed, keeping namedtuple field names."""
    fields = getattr(shape, '_fields', None)
    kept = tuple(d for d in shape if d > 1)
    if fields is None:
        return kept
    names = [f for f, d in zip(fields, shape) if d > 1]
    return namedtuple('SampleShape', names)(*kept)


class StreamBase:
    """State shared by readers and writers (base/base.py:409-599)."""

    _sample_shape_maker = None

    def __init__(self, fh_raw, header0, *, squeeze=True, device=None,
                 **kwargs):
        self.fh_raw = fh_raw
        self._header0 = header0
        self._squeeze = bool(squeeze)
        self._device_arg = device
        for attr, conv in (('bps', operator.index), ('complex_data', bool),
                           ('samples_per_frame', operator.index),
                           ('sample_shape', tuple), ('sample_rate', as_hertz)):
            value = kwargs.pop(attr, None)
            if value is None:
                value = getattr(header0, attr, None)
            if value is not None:
                value = conv(value)
            setattr(self, '_' + attr, value)
        if kwargs:
            raise TypeError('got unexpected keyword(s): {}'.format(
                ', '.join(kwargs)))
        if self._sample_rate is None:
            raise ValueError('the sample rate could not be determined; pass '
                             'in sample_rate explicitly.')
        self._frame_rate = self._sample_rate / self._samples_per_frame
        self.offset = 0
        self._closed = False

    # ---------------------------------------------------------------- props
    header0 = property(lambda self: self._header0)
    squeeze = property(lambda self: self._squeeze)
    bps = property(lambda self: self._bps)
    complex_data = property(lambda self: self._complex_data)
    samples_per_frame = property(lambda self: self._samples_per_frame)
    sample_rate = property(lambda self: self._sample_rate)

    @property
    def device(self):
        """CUDA device the samples are decoded / encoded on."""
        return _device.resolve(self._device_arg)

    @property
    def _unsliced_shape(self):
        if self._sample_shape_maker is not None:
            return self._sample_shape_maker(*self._sample_shape)
        return self._sample_shape

    @property
    def sample_shape(self):
        if '_sample_shape_cache' not in self.__dict__:
            shape = self._unsliced_shape
            self._sample_shape_cache = (_squeezed(shape) if self._squeeze
                                        else shape)
        return self._sample_shape_cache

    @property
    def dtype(self):
        return np.dtype(np.complex64 if self._complex_data else np.float32)

    # ---------------------------------------------------------------- time
    def _get_time(self, header):
        return header.time

    def _set_time(self, header, time):
        header.update(time=time)

    def _get_index(self, header):
        """Frame index of ``header`` relative to the first frame."""
        dt = self._get_time(header) - self.start_time
        return int(round(dt * self._frame_rate))

    def _set_index(self, header, index):
        self._set_time(header, self.start_time + index / self._frame_rate)

    @property
    def start_time(self):
        if '_start_time' not in self.__dict__:
            self._start_time = as_time(self._get_time(self.header0))
        return self._start_time

    @property
    def time(self):
        return self.tell(unit='time')

    def tell(self, unit=None):
        """Offset in samples (default), in a time unit ('s', 'ms', ...), or
        as absolute time (``unit='time'``)."""
        if unit is None:
            return self.offset
        if isinstance(unit, str) and unit == 'time':
            return self.start_time + self._offset_seconds(self.offset)
        scale = _TIME_UNITS.get(str(unit))
        if scale is None:
            raise ValueError('unknown time unit {!r}'.format(unit))
        return self.offset / self._sample_rate * scale

    def _offset_seconds(self, offset):
        from fractions import Fraction
        rate = Fraction(self._sample_rate).limit_denominator(10**9)
        return Fraction(offset) / rate

    # ----------------------------------------------------------- lifecycle
    @property
    def closed(self):
        return self._closed or getattr(self.fh_raw, 'closed', False)

    @property
    def name(self):
        return getattr(self.fh_raw, 'name', None)

    def readable(self):
        return hasattr(self, 'read') and not self.closed

    @property
    def info(self):
        """Basic stream properties as an info object (the reference's
        ``fh.info``, baseband/base/file_info.py:322-430, without its
        consistency checks)."""
        from .opener import FormatInfo
        fmt = type(self).__module__.split('.')[-2]
        attrs = dict(sample_rate=self.sample_rate,
                     sample_shape=tuple(self.sample_shape),
                     samples_per_frame=self.samples_per_frame,
                     bps=self.bps, complex_data=self.complex_data,
                     start_time=self.start_time, readable=self.readable())
        if hasattr(self, 'read'):
            attrs.update(shape=self.shape, stop_time=self.stop_time)
        return FormatInfo(fmt, True, **attrs)

    def writable(self):
        return hasattr(self, 'write') and not self.closed

    def seekable(self):
        return hasattr(self, 'seek') and not self.closed

    def close(self):
        self._closed = True
        close = getattr(self.fh_raw, 'close', None)
        if close is not None:
            close()

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc_val, exc_tb):
        self.close()

    def __repr__(self):
        return ('<{} name={} offset={}\n    sample_rate={} Hz, '
                'samples_per_frame={},\n    sample_shape={}, bps={},\n'
                '    start_time={}>'.format(
                    type(self).__name__, self.name, self.offset,
                    self.sample_rate, self.samples_per_frame,
                    self.sample_shape, self.bps, self.start_time.isot))


class _Stage:
    """One pipeline stage: pinned input, device input, device output."""

    def __init__(self):
        self.pin = None
        self.raw = None
        self.dec = None
        self.done = None          # event: stage's D2H (or H2D) finished
        self.free = None          # event: kernels no longer read ``raw``
        self.host = None          # pinned staging of the decoded output
        self.pending = None       # (host view, destination) still to copy

    def host_out(self, like):
        """Pinned staging tensor shaped and typed like the device tensor
        ``like``."""
        nbytes = like.numel() * like.element_size()
        if self.host is None or self.host.numel() < nbytes:
            self.host = _device.pinned_empty(nbytes, torch.uint8)
        return self.host[:nbytes].view(like.dtype).view(like.shape)

    def flush(self):
        """Finish a staged host copy: wait for the D2H into the pinned
        staging, then copy (several threads) into the caller's array."""
        if self.pending is None:
            return
        src, dst = self.pending
        self.pending = None
        self.done.synchronize()
        _device._threaded_copy(dst.reshape(-1).view(np.uint8),
                               src.numpy().reshape(-1).view(np.uint8))

    def buffers(self, nbytes, nfloat, dev, need_dec, dtype=torch.float32):
        if self.pin is None or self.pin.numel() < nbytes:
            self.pin = _device.pinned_empty(nbytes, torch.uint8)
            self.raw = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        if need_dec and (self.dec is None or self.dec.numel() < nfloat
                         or self.dec.dtype != dtype):
            self.dec = torch.empty(nfloat, dtype=dtype, device=dev)
        return self.pin[:nbytes], self.raw[:nbytes]


class StreamReaderBase(StreamBase):
    """Batched GPU stream reader.

    Subclasses provide the frame geometry (``_nframe``, ``_frame_nbytes``,
    ``_file_offset0``) and ``_decode_chunk``; everything else is here.

    Parameters beyond the reference's: ``device`` (CUDA device to decode on;
    when given, ``read`` returns a ``torch.Tensor`` on that device),
    ``chunk_nbytes`` (packed bytes per pipeline stage) and ``dtype``
    (``None`` / ``'float32'``: float32 / complex64 samples as the reference
    returns them; ``'float16'``: float16 / complex32; ``'bfloat16'``:
    bfloat16, complex samples with a trailing axis of 2 (re, im); torch dtypes
    are accepted too).  The kernels write the reduced types directly: every
    value is the float32 result rounded to nearest even, as ``.to(dtype)``
    rounds it.  With a reduced ``dtype``, ``read`` always returns a torch
    tensor (numpy has neither bfloat16 nor complex half): on ``device``, or
    in pinned host memory that the device-to-host copy lands in (small reads,
    sliced from the decoded window, in ordinary host memory).
    """

    def __init__(self, fh_raw, header0, *, squeeze=True, subset=(),
                 fill_value=0., verify=True, device=None,
                 chunk_nbytes=None, dtype=None, **kwargs):
        super().__init__(fh_raw, header0, squeeze=squeeze, device=device,
                         **kwargs)
        # the torch dtype the kernels write: float32, float16 or bfloat16
        self._dec_dtype = _decode_dtype_arg(dtype)
        if subset is None:
            subset = ()
        elif not isinstance(subset, tuple):
            subset = (subset,)
        self._subset = subset
        self._fill_value = float(fill_value)
        self.verify = verify
        self._device_output = device is not None
        self._chunk_nbytes = int(chunk_nbytes or DEFAULT_CHUNK_NBYTES)
        self._on_device = None
        self._stages = None
        self._streams = None
        self.sample_shape            # validates the subset

    subset = property(lambda self: self._subset)
    fill_value = property(lambda self: self._fill_value)

    @property
    def dtype(self):
        """Element type of what ``read`` returns: the numpy float32 /
        complex64 of the reference by default, else the torch dtype
        (float16, complex32 or bfloat16)."""
        if self._dec_dtype == torch.float32:
            return StreamBase.dtype.fget(self)
        return self._result_dtype(self._dec_dtype)

    def _result_dtype(self, dec):
        """torch dtype of the samples decoded as ``dec`` elements."""
        if not self._complex_data:
            return dec
        return {torch.float32: torch.complex64,
                torch.float16: torch.complex32}.get(dec, dec)

    def _pair_axis(self, dec):
        """(2,) where complex samples keep a (re, im) axis (bfloat16)."""
        return (2,) if self._complex_data and dec == torch.bfloat16 else ()

    def _read_decode_dtype(self, out):
        """Element type the kernels write for a read into ``out``: the
        reader's, except that a float32 reader handed a float16 / complex32 /
        (real) bfloat16 torch tensor decodes straight to it."""
        if self._dec_dtype == torch.float32 and isinstance(out, torch.Tensor):
            for dec in (torch.float16, torch.bfloat16):
                if (out.dtype == self._result_dtype(dec)
                        and not self._pair_axis(dec)):
                    return dec
        return self._dec_dtype

    def _complex_view(self, t):
        """Decoded (..., 2) elements -> complex samples (bfloat16: kept
        as they are)."""
        return t if t.dtype == torch.bfloat16 else torch.view_as_complex(t)

    # --------------------------------------------------------------- shapes
    @property
    def sample_shape(self):
        if '_sample_shape_cache' in self.__dict__:
            return self._sample_shape_cache
        shape = StreamBase.sample_shape.fget(self)
        if self._subset:
            # Index a dummy sample set to learn the resulting shape, checking
            # that sample numbers survive (base/base.py:720-776 behaviour).
            marks = np.arange(13.)
            dummy = np.moveaxis(np.zeros(tuple(shape))[..., np.newaxis]
                                + marks, -1, 0)
            try:
                picked = dummy[(slice(None),) + self._subset]
                assert 0 not in picked.shape
                assert np.all(np.moveaxis(picked, 0, -1) == marks)
            except (IndexError, AssertionError) as exc:
                exc.args += ('subset {} cannot be used to properly index '
                             '{}samples with shape {}.'.format(
                                 self._subset,
                                 'squeezed ' if self.squeeze else '',
                                 tuple(shape)),)
                self.__dict__.pop('_sample_shape_cache', None)
                raise
            shape = self._named_subset_shape(shape, picked.shape[1:])
        self._sample_shape_cache = shape
        return shape

    def _named_subset_shape(self, shape, subset_shape):
        fields = getattr(shape, '_fields', None)
        if (fields is None or subset_shape == ()
                or len(self._subset) > len(shape)):
            return subset_shape
        items = self._subset + (slice(None),) * (len(shape)
                                                 - len(self._subset))
        names, axis = [], 0
        try:
            for name, dim, item in zip(fields, shape, items):
                kept = np.empty(dim)[item].shape
                assert len(kept) <= 1
                if len(kept) == 1:
                    assert kept[0] == subset_shape[axis]
                    names.append(name)
                    axis += 1
        except Exception:
            return subset_shape
        return namedtuple('SampleShape', names)(*subset_shape)

    @property
    def _nsample(self):
        """Number of complete samples in the stream."""
        return self._nframe * self._samples_per_frame

    @property
    def shape(self):
        return (self._nsample,) + tuple(self.sample_shape)

    @property
    def size(self):
        return int(np.prod(self.shape))

    @property
    def ndim(self):
        return len(self.shape)

    @property
    def stop_time(self):
        return self.start_time + self._offset_seconds(self._nsample)

    # ----------------------------------------------------------- seek/tell
    def seek(self, offset, whence=0):
        """Move the sample pointer.  ``offset`` is a number of samples, a
        `~baseband_b200.timeutil.Time` (absolute; whence ignored) or a float
        number of seconds wrapped as ``('s', value)``."""
        if isinstance(offset, Time) or hasattr(offset, 'isot'):
            dt = as_time(offset) - self.start_time
            offset = int(round(dt * self._sample_rate))
            whence = 0
        elif isinstance(offset, tuple):
            unit, value = offset
            offset = int(round(value / _TIME_UNITS[unit] * self._sample_rate))
        else:
            try:
                offset = operator.index(offset)
            except TypeError:
                to_value = getattr(offset, 'to_value', None)
                if to_value is None:
                    raise
                offset = int(round(to_value('s') * self._sample_rate))
        if whence == 0 or whence == 'start':
            self.offset = offset
        elif whence == 1 or whence == 'current':
            self.offset += offset
        elif whence == 2 or whence == 'end':
            self.offset = self._nsample + offset
        else:
            raise ValueError("invalid 'whence'; should be 0 or 'start', 1 or "
                             "'current', or 2 or 'end'.")
        return self.offset

    # ----------------------------------------------------------------- read
    def read(self, count=None, out=None, *, on_device=None):
        """Read and decode ``count`` complete samples.

        Returns an array ``(count,) + sample_shape`` of float32/complex64:
        a `numpy.ndarray`, or a CUDA `torch.Tensor` if the stream was opened
        with ``device=`` or ``out`` is a CUDA tensor.  ``out`` may be a numpy
        array or a torch tensor whose leading dimension sets ``count``.  With
        a reduced ``dtype`` (see the class) the result is a torch tensor of
        that type; ``out`` is then a torch tensor of it, or, for real float16
        streams, also a numpy float16 array.

        ``on_device`` (extension): a callable that is handed every decoded
        chunk as a CUDA tensor ``(n,) + sample_shape``, in order, on the
        compute stream, before the chunk is copied to the host -- the hook
        for consumers that work on the GPU (e.g. ``writer.write`` to
        re-encode while the samples are still in HBM).
        """
        if self.closed:
            raise ValueError('I/O operation on closed file.')
        if out is None:
            if count is None or count < 0:
                count = max(0, self._nsample - self.offset)
        else:
            trailing = tuple(self.sample_shape) + self._pair_axis(
                self._dec_dtype)
            assert tuple(out.shape[1:]) == trailing, (
                "'out' must have trailing shape {}".format(trailing))
            if (isinstance(out, np.ndarray)
                    and self._dec_dtype != torch.float32
                    and (self.dtype != torch.float16
                         or out.dtype != np.float16)):
                raise TypeError('out must be a torch tensor of {}{}'.format(
                    self.dtype, ' or a numpy float16 array'
                    if self.dtype == torch.float16 else ''))
            count = out.shape[0]
        if count > 0 and (self.offset < 0
                          or self.offset + count > self._nsample):
            raise EOFError('cannot read from beyond end of input.')
        to_device = _device.is_device_tensor(out) or (
            out is None and self._device_output)
        if (not to_device and on_device is None and count > 0
                and self._small_read_cache_ok
                and (out is None or isinstance(out, np.ndarray))
                and count * self._floats_per_sample * self._dec_dtype.itemsize
                <= self.SMALL_READ_NBYTES):
            result = self._read_small_cached(self.offset, count, out)
            self.offset += count
            return result
        self._on_device = on_device
        try:
            if to_device:
                result = self._read_to_device(self.offset, count, out)
            else:
                result = self._read_to_host(self.offset, count, out)
        finally:
            self._on_device = None
        self.offset += count
        return result

    # Small host reads.  The reference decodes a whole frame and keeps it, so
    # a loop of small reads costs one decode per frame plus slicing
    # (base/base.py:990-996).  A GPU round trip per call (copy in, launch,
    # copy out: ~0.4 ms) would make exactly that pattern slower than the
    # reference, so small reads are served from a decoded window of whole
    # frames (at most SMALL_READ_WINDOW_NBYTES), refilled when a read leaves it.
    SMALL_READ_NBYTES = 256 << 10
    SMALL_READ_WINDOW_NBYTES = 8 << 20
    _small_cache = None
    # False where the samples returned depend on where a read starts (GUPPI
    # frames with overlap: a read runs on through the overlap of the frame it
    # starts in, guppi/base.py:203-221)
    _small_read_cache_ok = True

    def _read_small_cached(self, start, count, out):
        nb = self._floats_per_sample * self._dec_dtype.itemsize
        block = max(1, min(self._samples_per_frame,
                           self.SMALL_READ_WINDOW_NBYTES // nb))
        cache = self._small_cache
        if (cache is None or start < cache[0] or start + count > cache[1]
                or cache[3] != self._fill_value):
            w0 = start // block * block
            w1 = min(self._nsample, -(-(start + count) // block) * block)
            data = self._read_to_host(w0, w1 - w0, None)
            cache = self._small_cache = (w0, w1, data, self._fill_value)
        piece = cache[2][start - cache[0]:start - cache[0] + count]
        if out is None:
            return piece.clone() if isinstance(piece, torch.Tensor) \
                else piece.copy()
        out[...] = piece
        return out

    # -- geometry hooks --------------------------------------------------
    _file_offset0 = 0            # byte offset of frame 0 in the file

    def _frame_span(self, start, count):
        """Frames [f0, f1) holding samples [start, start + count)."""
        spf = self._samples_per_frame
        return start // spf, -(-(start + count) // spf)

    def _frame_sample0(self, frame):
        """Stream sample number of the first sample of ``frame``."""
        return frame * self._samples_per_frame

    def _frames_per_chunk(self):
        return max(1, self._chunk_nbytes // self._frame_nbytes)

    # Irregular streams (missing / duplicated / re-ordered frames, bytes
    # lost or inserted between frames): a reader may install ``_index``, an
    # int64 table (nframe, nslot) of the BYTE OFFSETS of the frames in the
    # file (-1 = absent), built on the device by `_build_index_on_device`.
    # Chunks are then read as the byte span of the frames they touch.
    _index = None

    def _set_index_table(self, table, phys_frame_nbytes):
        self._small_cache = None     # decoded without the index: stale
        self._layout_cache = None
        self._index = table
        self._index_lo = np.where(table >= 0, table,
                                  np.iinfo(np.int64).max)
        self._phys_frame_nbytes = phys_frame_nbytes
        self._nframe = table.shape[0]

    def _chunk_first_byte(self, frame0, nframe):
        """File offset of the first frame a chunk touches."""
        lo = self._index_lo[frame0:frame0 + nframe].min()
        return 0 if lo == np.iinfo(np.int64).max else int(lo)

    def _chunk_nbytes_of(self, frame0, nframe, sample_start, nsample):
        """Raw bytes a chunk needs on the device (and in pinned memory)."""
        if self._index is None:
            return nframe * self._frame_nbytes
        _, span, dev_nbytes, _, _ = self._chunk_layout(frame0, nframe)
        return max(span, dev_nbytes)

    _layout_cache = None

    def _chunk_layout(self, frame0, nframe):
        """How the frames of an indexed chunk get to the device:
        ``(first_byte, span, dev_nbytes, runs, rel)``.  The file bytes
        [first_byte, first_byte + span) hold every frame of the chunk.  Where
        all frames sit a multiple of 16 bytes from the first (whole frames
        missing or re-ordered), that span goes up in one copy.  Bytes lost or
        inserted between frames shift the later ones off the kernels' word
        alignment: the span is then copied as ``runs`` of equally aligned
        frames ``(source offset, device offset, length)``, each to a 16-byte
        boundary.  ``rel`` (nframe, nslot) = device offset of each frame in
        the chunk buffer, -1 where absent."""
        key = (frame0, nframe)
        if self._layout_cache is not None and self._layout_cache[0] == key:
            return self._layout_cache[1]
        fb = self._phys_frame_nbytes
        table = self._index[frame0:frame0 + nframe]
        valid = table >= 0
        first = self._chunk_first_byte(frame0, nframe)
        rel = np.full(table.shape, -1, np.int64)
        if not valid.any():
            layout = (first, fb, fb, [(0, 0, fb)], rel)
        else:
            offs = np.unique(table[valid])               # file order
            span = int(offs[-1]) + fb - first
            phase = (offs - first) % 16
            if not phase.any():
                rel[valid] = table[valid] - first
                layout = (first, span, span, [(0, 0, span)], rel)
            else:
                breaks = np.flatnonzero(np.diff(phase)) + 1
                starts = np.concatenate([[0], breaks])
                stops = np.concatenate([breaks, [offs.size]])
                shift = np.empty(offs.size, np.int64)
                runs, dst = [], 0
                for a, b in zip(starts, stops):
                    src = int(offs[a]) - first
                    length = int(offs[b - 1]) + fb - int(offs[a])
                    runs.append((src, dst, length))
                    shift[a:b] = dst - src
                    dst += -(-length // 16) * 16
                at = np.searchsorted(offs, table[valid])
                rel[valid] = table[valid] - first + shift[at]
                layout = (first, span, dst, runs, rel)
        self._layout_cache = (key, layout)
        return layout

    def _upload(self, raw, pin, frame0, nframe):
        """Queue the host-to-device copy of a chunk on the current stream."""
        if self._index is None:
            raw.copy_(pin, non_blocking=True)
            return
        _, _, _, runs, _ = self._chunk_layout(frame0, nframe)
        for src, dst, length in runs:
            raw[dst:dst + length].copy_(pin[src:src + length],
                                        non_blocking=True)

    def _build_index_on_device(self, pattern, mask, frame_nbytes,
                               index_chunk, nslot, nset_max,
                               pattern_offset=0):
        """Frame table of an irregular stream, built on the GPU: the file is
        streamed through the device in overlapping chunks; in each,
        bb_locate_frames finds every place the stream's (masked) sync pattern
        starts a frame that is followed by another one (or the end of the
        file) -- the reference's `locate_frames` (base/base.py:181-335) over
        the whole file -- and ``index_chunk(raw, base, locations, count,
        table, stats)`` scatters the frames found into the table by their
        header time (bb_vdif_index / bb_mark5b_index).  Returns the table
        (nset, nslot) of byte offsets on the host and the kernels' stats."""
        from .. import kernels
        dev = self.device
        fh = self.fh_raw
        size = fh.seek(0, 2)
        fh.seek(0)
        pat = kernels._host_bytes(pattern)[0]
        msk = kernels._host_bytes(mask)[0]
        overlap = frame_nbytes + pattern_offset + pat.size
        step = max(4 * frame_nbytes, self._chunk_nbytes // frame_nbytes
                   * frame_nbytes)
        table = kernels.index_table(nset_max * nslot, dev)
        stats = kernels.zeros(4, torch.int32, dev)
        counts = []
        # headers not followed by another one (kept aside, see below)
        loose = (torch.empty(4096, dtype=torch.int64, device=dev),
                 kernels.zeros(1, torch.int32, dev))
        stages, ss = self._pipeline(dev)
        zero_copy = getattr(fh, 'pinned_view', None)
        ss.after_caller(1)
        pos, k = self._file_offset0, 0
        while pos < size:
            n = min(step + overlap, size - pos)
            at_eof = pos + n >= size
            st = stages[k % 2]
            if st.done is not None:
                st.done.synchronize()
            pin, raw = st.buffers(n, 0, dev, False)
            view = zero_copy(pos, n) if zero_copy is not None else None
            if view is None:
                got = read_file_into(fh, pos, pin.numpy())
                if got != n:
                    raise EOFError('could not read the file for indexing.')
                view = pin
            with ss.use(0):
                ss.wait_event(0, st.free)
                raw.copy_(view, non_blocking=True)
                st.done = ss.event(0)
            with ss.use(1):
                ss.wait_event(1, st.done)
                locations, count = kernels.locate_frames(
                    raw, pat, msk, frame_nbytes, pattern_offset,
                    own_stop=n if at_eof else step, check=1, at_eof=at_eof,
                    base=pos, unverified=loose)
                index_chunk(raw, pos, locations, count, table, stats)
                st.free = ss.event(1)
            counts.append((count, locations.numel()))
            if at_eof:
                break
            pos += step
            k += 1
        with ss.use(1):
            offsets = kernels.index_table_finish(table)
        ss.caller_after(1)
        if any(int(count.item()) > room for count, room in counts):
            raise OSError('too many sync-pattern candidates to index this '
                          'file: is it in this format at all?')
        stats = stats.cpu().numpy()
        nset = int(stats[0]) + 1
        host = offsets[:nset * nslot].cpu().numpy().reshape(nset, nslot)
        if not (host >= 0).any():
            host = host[:0]
        nloose = min(int(loose[1].item()), loose[0].numel())
        self._index_loose = np.sort(loose[0][:nloose].cpu().numpy())
        return host, stats

    def _read_raw(self, frame0, nframe, pinned, sample_start=0, nsample=0):
        """Fill ``pinned`` (uint8 tensor) with the bytes of frames
        [frame0, frame0 + nframe)."""
        if self._index is not None:
            offset, span = self._chunk_layout(frame0, nframe)[:2]
            pinned = pinned[:span]
        else:
            offset = self._file_offset0 + frame0 * self._frame_nbytes
        zero_copy = getattr(self.fh_raw, 'pinned_view', None)
        if zero_copy is not None:
            # frames already sit in pinned host memory: no staging copy
            view = zero_copy(offset, pinned.numel())
            if view is not None:
                return view
        view = pinned.numpy()
        got = read_file_into(self.fh_raw, offset, view)
        if got != view.size:
            raise EOFError('could not read {} frames at frame {}.'.format(
                nframe, frame0))
        return pinned

    def _read_raw_begin(self, frame0, nframe, pinned, sample_start=0,
                        nsample=0):
        """Start filling ``pinned`` with the bytes of a chunk and return a
        handle whose ``wait()`` gives the tensor to upload.  For plain files
        the copy out of the page cache runs on the library's thread pool
        while the caller queues the previous chunk's GPU work (one chunk of
        read-ahead); everything else is read on the spot."""
        if (type(self)._read_raw is StreamReaderBase._read_raw
                and PARALLEL_READ_MMAP and PARALLEL_READ_THREADS >= 1
                and getattr(self.fh_raw, 'pinned_view', None) is None):
            if self._index is not None:
                offset, span = self._chunk_layout(frame0, nframe)[:2]
                target = pinned[:span]
            else:
                offset = self._file_offset0 + frame0 * self._frame_nbytes
                target = pinned
            n = target.numel()
            plain = _plain_file(self.fh_raw)
            if plain is not None and n >= PARALLEL_READ_MIN_NBYTES:
                mapped = _mapped_file(plain[0], plain[1], offset + n)
                if mapped is not None and mapped[1].size >= offset + n:
                    import ctypes
                    from .._lib import host_io
                    lib = host_io()
                    rc = lib.bb_host_copy_begin(
                        ctypes.c_void_p(target.data_ptr()),
                        ctypes.c_void_p(mapped[1].ctypes.data + offset), n,
                        PARALLEL_READ_THREADS)
                    if rc == 0:
                        return _PendingCopy(lib, target, n)
        got = self._read_raw(frame0, nframe, pinned, sample_start, nsample)
        return _Ready(pinned if got is None else got)

    def _decode_chunk(self, raw, frame0, nframe, sample_start, nsample, out):
        """Decode ``nsample`` samples starting ``sample_start`` samples into
        the first frame of ``raw`` (device bytes of ``nframe`` frames) into
        the float32, float16 or bfloat16 device tensor ``out`` (flat,
        unsliced sample layout)."""
        raise NotImplementedError

    # -- helpers ---------------------------------------------------------
    @property
    def _floats_per_sample(self):
        n = 2 if self._complex_data else 1
        for dim in self._unsliced_shape:
            n *= dim
        return n

    def _finish(self, flat, nsample):
        """Decoded device buffer -> (nsample, *sample_shape) tensor."""
        shape = tuple(self._unsliced_shape)
        if self._complex_data:
            data = self._complex_view(
                flat[:nsample * self._floats_per_sample].view(
                    (nsample,) + shape + (2,)))
        else:
            data = flat[:nsample * self._floats_per_sample].view(
                (nsample,) + shape)
        return self._squeeze_and_subset(data)

    def _squeeze_and_subset(self, data):
        if self._squeeze:
            data = data.reshape(tuple(data.shape[:1]) + tuple(
                d for d in data.shape[1:] if d > 1))
        if self._subset:
            data = data[(slice(None),) + _torch_index(self._subset,
                                                      data.device)]
        return data

    def _chunks(self, start, count):
        """Yield (frame0, nframe, sample_start, nsample, row0)."""
        if count == 0:
            return
        f0, f1 = self._frame_span(start, count)
        per = self._frames_per_chunk()
        row = 0
        for c0 in range(f0, f1, per):
            c1 = min(c0 + per, f1)
            first = max(start, self._frame_sample0(c0))
            last = (start + count if c1 == f1
                    else min(start + count, self._frame_sample0(c1)))
            yield c0, c1 - c0, first - self._frame_sample0(c0), last - first, row
            row += last - first

    # Frame-regularity checks are folded into the scan kernels, which add to
    # one device counter per reader; a read looks at it once, at its end.
    _bad_dev = None
    _bad_seen = 0
    _bad_dirty = False

    def _bad_counter(self, dev):
        """The counter, for a scan that is about to be launched."""
        if self._bad_dev is None or self._bad_dev.device != dev:
            from .. import kernels
            self._bad_dev = kernels.new_counter(dev)
            self._bad_seen = 0
        self._bad_dirty = True
        return self._bad_dev

    def _new_inconsistencies(self):
        """Frames the scan kernels found out of place since the last call
        (synchronises with the device, but only if a scan ran since)."""
        if self._bad_dev is None or not self._bad_dirty:
            return 0
        self._bad_dirty = False
        now = int(self._bad_dev.item())
        new, self._bad_seen = now - self._bad_seen, now
        return new

    def _pipeline(self, dev):
        """The pipeline stages and streams.  Host-output reads and the index
        build alternate between the first two stages; reads that leave their
        result on the device (and the packed consumers) rotate over all
        three, so that starting the read-ahead of chunk k + 1 never has to
        wait for the upload of chunk k - 1 to release its pinned buffer --
        with two, the next upload was only queued after that wait, and the
        copy engine idled for a host wake-up between chunks."""
        if self._stages is None:
            self._stages = [_Stage() for _ in range(3)]
            self._streams = _device.Streams(dev)
        return self._stages, self._streams

    # -- packed consumers ------------------------------------------------
    def _packed_units(self, raw, frame0, nframe):
        """Unit table of a chunk for consumers that work on the packed
        payloads: ``(unit_offset, nthread, payload_nbytes, bps, nelem)`` as
        the bit-field kernels take them.  Formats whose payloads are not
        plain bit fields do not provide it."""
        raise NotImplementedError('{} has no packed bit-field payloads'
                                  .format(type(self).__name__))

    def _for_each_packed_chunk(self, frame0, nframe, fn):
        """Stream the raw bytes of frames [frame0, frame0 + nframe) through
        the device -- the reader's own ingest pipeline: pinned (or zero-copy)
        host chunk -> H2D on the copy stream, double buffered -- and call
        ``fn(raw, first_frame, nframe_in_chunk)`` for every chunk on the
        compute stream.  Nothing is decoded."""
        dev = self.device
        stages, ss = self._pipeline(dev)
        spf = self._samples_per_frame
        per = self._frames_per_chunk()
        ss.after_caller(1)
        starts = list(range(frame0, frame0 + nframe, per))

        def begin(k):
            c0 = starts[k]
            nf = min(per, frame0 + nframe - c0)
            st = stages[k % DEVICE_READ_STAGES]
            if st.done is not None:
                st.done.synchronize()
            pin, _ = st.buffers(self._chunk_nbytes_of(c0, nf, 0, nf * spf),
                                0, dev, False)
            return self._read_raw_begin(c0, nf, pin, 0, nf * spf)

        ahead = begin(0) if starts else None
        for k, c0 in enumerate(starts):
            nf = min(per, frame0 + nframe - c0)
            st = stages[k % DEVICE_READ_STAGES]
            raw = st.raw[:self._chunk_nbytes_of(c0, nf, 0, nf * spf)]
            pin = ahead.wait()
            ahead = begin(k + 1) if k + 1 < len(starts) else None
            try:
                with ss.use(0):
                    ss.wait_event(0, st.free)
                    self._upload(raw, pin, c0, nf)
                    st.done = ss.event(0)
                with ss.use(1):
                    ss.wait_event(1, st.done)
                    fn(raw, c0, nf)
                    st.free = ss.event(1)
            except BaseException:
                if ahead is not None:
                    ahead.wait()
                raise
        ss.caller_after(1)

    # -- device output ---------------------------------------------------
    def _read_to_device(self, start, count, out):
        dev = out.device if out is not None else self.device
        fps = self._floats_per_sample
        dec = self._read_decode_dtype(out)
        direct = (out is not None and not self._subset and out.is_contiguous()
                  and out.dtype == self._result_dtype(dec))
        if direct:
            flat = (torch.view_as_real(out) if out.is_complex()
                    else out).reshape(-1)
        else:
            flat = torch.empty(count * fps, dtype=dec, device=dev)
        stages, ss = self._pipeline(dev)
        ss.after_caller(1)
        chunks = list(self._chunks(start, count))

        def begin(k):
            """Start reading chunk k into its stage's pinned buffer."""
            f0, nf, s0, ns, _ = chunks[k]
            st = stages[k % DEVICE_READ_STAGES]
            if st.done is not None:
                st.done.synchronize()        # pinned buffer free again
            pin, _ = st.buffers(self._chunk_nbytes_of(f0, nf, s0, ns), 0,
                                dev, False)
            return self._read_raw_begin(f0, nf, pin, s0, ns)

        ahead = begin(0) if chunks else None
        for k, (f0, nf, s0, ns, row) in enumerate(chunks):
            st = stages[k % DEVICE_READ_STAGES]
            raw = st.raw[:self._chunk_nbytes_of(f0, nf, s0, ns)]
            pin = ahead.wait()
            # the next chunk leaves the page cache while this one's copy and
            # kernels are queued
            ahead = begin(k + 1) if k + 1 < len(chunks) else None
            try:
                self._queue_chunk(ss, st, raw, pin, flat, fps, dev,
                                  f0, nf, s0, ns, row)
            except BaseException:
                if ahead is not None:
                    ahead.wait()
                raise
        ss.caller_after(1)
        result = self._finish(flat, count)
        if out is not None and not direct:
            out.copy_(result)
            return out
        return out if direct else result

    def _queue_chunk(self, ss, st, raw, pin, flat, fps, dev, f0, nf, s0, ns,
                     row):
        """H2D copy and decode of one chunk of a device-output read."""
        with ss.use(0):
            # raw[k%2] must no longer be read by the decode of chunk k-2
            # (only that: the copy overlaps the decode of chunk k-1)
            ss.wait_event(0, st.free)
            self._upload(raw, pin, f0, nf)
            st.done = ss.event(0)
        with ss.use(1):
            ss.wait_event(1, st.done)
            piece = flat[row * fps:(row + ns) * fps]
            # the kernels store 4 elements at a time (16 / 8 bytes)
            if piece.data_ptr() % (4 * piece.element_size()):
                tmp = torch.empty(ns * fps, dtype=piece.dtype, device=dev)
                self._decode_chunk(raw, f0, nf, s0, ns, tmp)
                piece.copy_(tmp)
            else:
                self._decode_chunk(raw, f0, nf, s0, ns, piece)
            if self._on_device is not None:
                self._on_device(self._finish(piece, ns))
            st.free = ss.event(1)

    # -- host output -----------------------------------------------------
    def _read_to_host(self, start, count, out):
        dev = self.device
        fps = self._floats_per_sample
        dec = self._read_decode_dtype(out)
        shape = (count,) + tuple(self.sample_shape) + self._pair_axis(dec)
        t_dtype = self._result_dtype(dec)
        reduced = dec != torch.float32
        staged = False
        if out is None:
            # The result itself is pinned memory: D2H lands in it directly.
            holder = (_device.pinned_empty(shape, t_dtype) if count > 0
                      else torch.empty(shape, dtype=t_dtype))
            target = holder
            result = holder if reduced else holder.numpy()
        elif isinstance(out, torch.Tensor):
            target, result = out, out
        else:
            result = out
            target = _as_host_tensor(out, np.dtype(np.float16) if reduced
                                     else self.dtype)
            # A large pageable destination: page-locking it in place costs
            # more than it saves (cudaHostRegister pins ~10 GB/s), so each
            # chunk lands in the stage's pinned buffer and is copied on by a
            # few threads while the next chunk is in flight.
            staged = (target is not None and not target.is_pinned()
                      and out.nbytes >= STAGED_HOST_OUT_MIN_NBYTES)
        if count == 0:
            return result
        stages, ss = self._pipeline(dev)
        try:
            for k, (f0, nf, s0, ns, row) in enumerate(
                    self._chunks(start, count)):
                st = stages[k % 2]
                nbytes = self._chunk_nbytes_of(f0, nf, s0, ns)
                st.flush()
                if st.done is not None:
                    st.done.synchronize()
                pin, raw = st.buffers(nbytes, ns * fps, dev, True, dec)
                got = self._read_raw(f0, nf, pin, s0, ns)
                pin = pin if got is None else got
                with ss.use(0):
                    self._upload(raw, pin, f0, nf)
                with ss.use(1):
                    ss.wait(1, 0)
                    self._decode_chunk(raw, f0, nf, s0, ns, st.dec[:ns * fps])
                    piece = self._finish(st.dec, ns)
                    if self._on_device is not None:
                        self._on_device(piece)
                    if self._subset and not piece.is_contiguous():
                        piece = piece.contiguous()
                    if piece.untyped_storage().data_ptr() \
                            != st.dec.untyped_storage().data_ptr():
                        # a fresh tensor (subset gather / contiguous copy)
                        # allocated under stream 1 but read by the D2H copy
                        # on stream 2: keep its block out of stream 1's pool
                        # until that copy is done
                        ss.keep_alive(piece, 2)
                with ss.use(2):
                    ss.wait(2, 1)
                    if staged:
                        hostbuf = st.host_out(piece)
                        hostbuf.copy_(piece, non_blocking=True)
                        st.pending = (hostbuf, result[row:row + ns])
                    elif target is not None:
                        target[row:row + ns].copy_(piece, non_blocking=True)
                    else:
                        # exotic ``out`` (wrong dtype / non-contiguous)
                        out[row:row + ns] = piece.cpu().numpy()
                    st.done = ss.event(2)
                # the other stage's chunk: its D2H has had a whole chunk's
                # time; copy it on while this chunk is in flight
                stages[(k + 1) % 2].flush()
            for st in stages:
                st.flush()
                if st.done is not None:
                    st.done.synchronize()
        finally:
            for st in stages:
                st.pending = None        # nothing stale after an error
        return result

    # Pickling (base/base.py:123-151, :1020-1032): device buffers and streams
    # are dropped and re-created lazily; the raw file is re-opened by name in
    # the unpickling process and the sample pointer restored.
    def __getstate__(self):
        state = self.__dict__.copy()
        state['_stages'] = None
        state['_streams'] = None
        state['_small_cache'] = None
        state.pop('_slots_dev', None)
        state.pop('_bad_dev', None)
        state.pop('_bad_seen', None)
        state.pop('_bad_dirty', None)
        state.pop('_sample_shape_cache', None)    # namedtuple made on the fly
        wrapper = state['fh_raw']
        fh = getattr(wrapper, 'fh_raw', wrapper)
        name = getattr(fh, 'name', None)
        if isinstance(name, str) and not getattr(fh, 'closed', False):
            import copy
            clone = copy.copy(wrapper) if fh is not wrapper else None
            state['fh_raw'] = ('__reopen__', name, clone)
            if clone is not None:
                clone.fh_raw = None
        return state

    def __setstate__(self, state):
        marker = state.get('fh_raw')
        if isinstance(marker, tuple) and marker and marker[0] == '__reopen__':
            _, name, clone = marker
            import io
            fh = io.open(name, 'rb')
            if clone is not None:
                clone.fh_raw = fh
                fh = clone
            state['fh_raw'] = fh
        self.__dict__.update(state)
        if '_slots_host' in state:
            self._slots_dev = None


_DECODE_DTYPES = {None: torch.float32, 'float32': torch.float32,
                  torch.float32: torch.float32, 'float16': torch.float16,
                  torch.float16: torch.float16, 'bfloat16': torch.bfloat16,
                  torch.bfloat16: torch.bfloat16}


def _decode_dtype_arg(dtype):
    """The reader's ``dtype`` argument -> torch dtype the kernels write."""
    try:
        return _DECODE_DTYPES[dtype]
    except (KeyError, TypeError):
        raise ValueError("dtype must be None, 'float32', 'float16' or "
                         "'bfloat16' (or the torch dtype), not {!r}"
                         .format(dtype)) from None


def _torch_index(subset, dev):
    out = []
    for item in subset:
        if isinstance(item, (list, np.ndarray)):
            item = torch.as_tensor(np.asarray(item), device=dev)
        out.append(item)
    return tuple(out)


def _as_host_tensor(arr, dtype):
    """A torch view of a numpy array if it can be a D2H target."""
    if not isinstance(arr, np.ndarray) or arr.dtype != dtype \
            or not arr.flags.c_contiguous or not arr.flags.writeable:
        return None
    return torch.from_numpy(arr)


class StreamWriterBase(StreamBase):
    """Batched GPU stream writer.

    ``write(data, valid=True)`` accepts numpy arrays or CUDA tensors of shape
    ``(n,) + sample_shape``.  Samples are collected until at least one whole
    frame is available; all whole frames are then quantised, packed and given
    headers in one pass (one encode kernel), copied back and written to the
    file (base/base.py:1276-1342 semantics, including the zero-padded,
    invalid last frame emitted by ``close``).

    torch tensors, on the device or on the host, may also hold the
    half-precision types a ``dtype=`` reader returns: float16 or bfloat16
    for real streams; complex32, or bfloat16 with a trailing (re, im) axis
    of 2, for complex streams.  They go to the device at 2 bytes per
    component and are encoded from there: each value gives exactly the bits
    its float32 value would.  Writes of mixed types are combined in
    ``torch.result_type`` of all of them (float16 with float32 or bfloat16
    gives float32, exactly; anything with float64 gives float64).  numpy
    float16 arrays are converted to float64, like other numpy types.

    Subclasses implement ``_encode_frames``.
    """

    def __init__(self, fh_raw, header0, *, squeeze=True, device=None,
                 **kwargs):
        super().__init__(fh_raw, header0, squeeze=squeeze, device=device,
                         **kwargs)
        self._pending = []           # [(tensor (n, fps...), valid)]
        self._nowned = 0             # leading entries that are our own copies
        self._npending = 0
        self._frame_index = 0

    def _pair(self, t):
        """Whether ``t`` holds complex samples as a trailing (re, im) axis."""
        return self._complex_data and not t.is_complex()

    def _unsqueeze(self, data):
        shape = tuple(self._unsliced_shape)
        pair = (2,) if self._pair(data) else ()
        given = tuple(data.shape[1:len(data.shape) - len(pair)])
        if given != shape:
            try:
                data = data.reshape((data.shape[0],) + shape + pair)
            except (RuntimeError, ValueError):
                raise ValueError('cannot reshape data with sample shape {} '
                                 'to {}'.format(given, shape))
        return data

    def _to_device(self, data):
        dev = self.device
        if isinstance(data, torch.Tensor):
            # 16-bit complex samples are kept as (re, im) pairs
            if self._complex_data and data.dtype == torch.complex32:
                # its float16 view: no other ComplexHalf op is needed
                return torch.view_as_real(data).to(dev)
            if self._complex_data and data.dtype == torch.bfloat16:
                if data.ndim < 2 or data.shape[-1] != 2:
                    raise ValueError('stream holds complex data: bfloat16 '
                                     'values need a trailing (re, im) axis '
                                     'of length 2')
                return data.to(dev)
            t = data.to(dev)
        else:
            arr = np.asanyarray(data)
            if arr.dtype.kind == 'c':
                arr = arr.astype(np.complex64 if arr.dtype.itemsize <= 8
                                 else np.complex128, copy=False)
            elif arr.dtype not in (np.float32, np.float64):
                arr = arr.astype(np.float64)
            arr = np.ascontiguousarray(arr)
            if arr.nbytes >= _device.STAGED_UPLOAD_MIN_NBYTES:
                t = _device.staged_upload(arr, dev)
            else:
                t = torch.from_numpy(arr).to(dev)
        if t.is_complex() != self._complex_data:
            if self._complex_data:
                raise ValueError('stream holds complex data but real values '
                                 'were given')
            raise ValueError('stream holds real data but complex values '
                             'were given')
        return t

    # Large host arrays are sent to the GPU in slices of this many bytes, so
    # device memory holds one slice, not the whole array; each slice goes
    # through `device.staged_upload` (threaded copy into pinned staging,
    # overlapped with the PCIe transfer).
    HOST_WRITE_SLICE_NBYTES = 256 << 20

    def write(self, data, valid=True):
        if self.closed:
            raise ValueError('I/O operation on closed file.')
        if isinstance(data, np.ndarray) and data.ndim >= 1 \
                and data.nbytes >= 2 * self.HOST_WRITE_SLICE_NBYTES:
            rows = max(1, self.HOST_WRITE_SLICE_NBYTES
                       // max(1, data.nbytes // data.shape[0]))
            for lo in range(0, data.shape[0], rows):
                self._write_one(data[lo:lo + rows], valid)
            return
        self._write_one(data, valid)

    def _write_one(self, data, valid):
        t = self._unsqueeze(self._to_device(data))
        if t.shape[0] == 0:
            return
        self._pending.append((t, bool(valid)))
        self._npending += t.shape[0]
        self.offset += t.shape[0]
        self._flush(final=False)

    def _flush(self, final):
        spf = self._samples_per_frame
        nframe = self._npending // spf
        if final and self._npending % spf:
            import warnings
            pad = spf - self._npending % spf
            warnings.warn('closing with partial buffer remaining.  Writing '
                          'padded frame, marked as invalid.')
            like = self._pending[-1][0]
            self._pending.append((torch.zeros((pad,) + tuple(like.shape[1:]),
                                              dtype=like.dtype,
                                              device=like.device), False))
            self._npending += pad
            nframe += 1
        if nframe == 0:
            # keep our own copy of what this call added: the caller's tensor
            # may be a view of a buffer that is about to be reused
            # (read(on_device=...)); earlier entries already are copies
            self._pending[self._nowned:] = [
                (t.clone(), ok) for t, ok in self._pending[self._nowned:]]
            self._nowned = len(self._pending)
            return
        take = nframe * spf
        # validity per frame = AND over the writes that touch it
        valid = np.ones(nframe, bool)
        pos = 0
        for t, ok in self._pending:
            n = t.shape[0]
            if not ok:
                a, b = pos // spf, min(nframe, -(-(pos + n) // spf))
                valid[a:b] = False
            pos += n
            if pos >= take:
                break
        pending = [t for t, _ in self._pending]
        if self._complex_data and any(self._pair(t) for t in pending):
            # 16-bit complex samples are kept as (re, im) pairs: combine all
            # in that form, so the types promote as their components do
            pending = [torch.view_as_real(t) if t.is_complex() else t
                       for t in pending]
        dtypes = {t.dtype for t in pending}
        dtype = functools.reduce(torch.promote_types, dtypes)
        data = torch.cat([t.to(dtype) for t in pending]) \
            if len(pending) > 1 else pending[0]
        rest = data[take:]
        rest_valid = self._pending[-1][1]
        data = data[:take].contiguous()
        if data.is_complex():
            data = torch.view_as_real(data)
        if data.element_size() == 2 and data.data_ptr() % 8:
            data = data.clone()          # the 16-bit loads need 8 bytes
        frames = self._encode_frames(data.reshape(-1), self._frame_index,
                                     nframe, valid)
        self._write_raw(frames)
        self._frame_index += nframe
        self._pending = [(rest.clone(), rest_valid)] if rest.shape[0] else []
        self._nowned = len(self._pending)
        self._npending = int(rest.shape[0])

    def _encode_frames(self, flat, index0, nframe, valid):
        """Return a uint8 CUDA tensor holding ``nframe`` complete frames
        (headers + encoded payloads) for samples ``flat`` (real view)."""
        raise NotImplementedError

    def _write_raw(self, frames):
        reserve = getattr(self.fh_raw, 'reserve', None)
        if reserve is not None:
            # sink is pinned host memory: let the D2H copy land in it
            reserve(frames.numel()).copy_(frames.view(-1), non_blocking=True)
            defer = getattr(self.fh_raw, 'defer', None)
            if defer is not None and frames.is_cuda:
                # the sink waits for the copy when its bytes are looked at;
                # the host goes on (inside read(on_device=writer.write) this
                # keeps the device-to-host link busy with the decoded chunk)
                defer(_device.record_event(frames.device))
            else:
                _device.current_stream_synchronize(frames.device)
            return
        host = _device.pinned_empty(frames.shape, torch.uint8)
        host.copy_(frames, non_blocking=True)
        _device.current_stream_synchronize(frames.device)
        self.fh_raw.write(memoryview(host.numpy()))

    def close(self):
        if not self._closed and self._npending:
            self._flush(final=True)
        super().close()
