"""Consumers that run on the GPU behind the stream readers.

The reference hands decoded samples to analysis code through the
``baseband.tasks`` plug-in point (baseband/tasks/__init__.py:25-62; the
baseband-tasks package: ``Square``, ``Integrate``, ...).  With the decode on
the GPU the end-to-end rate of ``fh.read()`` into host memory is set by the
device-to-host link (4 bytes per sample); a consumer that stays on the device
is not.  The ones here go one step further and never decode at all: they run
on the packed payloads as they arrive in HBM, through the reader's own ingest
pipeline (file / pinned host -> H2D -> header scan), and return a few numbers.

``state_counts(fh, samples_per_bin)``
    how often each code (state) occurs per integration bin, VDIF thread and
    channel -- the digitiser statistics -- as exact integers;
``integrated_power(fh, samples_per_bin)``
    mean (or summed) power per bin, thread and channel, the result of
    ``Integrate(Square(fh), samples_per_bin)``, from the same counts:
    ``sum(x**2) = sum_c counts[c] * level[c]**2``.  Invalid frames do not
    contribute (and do not count in the mean).

``moments(fh, samples_per_bin)``
    count, sum and sum of squares for 8-bit two's-complement streams (GUPPI),
    which `integrated_power` uses for those.

`state_counts` takes any reader with packed payloads: bit fields of 1, 2 or
4 bits (VDIF, Mark 5B, Mark 4, 4-bit GSB) and 8-bit samples (VDIF, GUPPI,
DADA, GSB phased), whose 256 states are counted by the stored byte.
"""
import numpy as np
import torch

from . import kernels

__all__ = ['state_counts', 'moments', 'integrated_power', 'state_levels']


def _frame_range(fh, count, samples_per_bin):
    spf = fh.samples_per_frame
    start = fh.tell()
    if count is None:
        count = fh.shape[0] - start
    if start % spf or count % spf:
        raise ValueError('state counts work on whole frames: the sample '
                         'pointer and count must be multiples of '
                         'samples_per_frame ({})'.format(spf))
    if count <= 0:
        raise ValueError('nothing to count')
    if samples_per_bin is None:
        samples_per_bin = count
    if samples_per_bin % spf:
        raise ValueError('samples_per_bin must be a multiple of '
                         'samples_per_frame ({})'.format(spf))
    return start // spf, count // spf, samples_per_bin // spf


def _units(fh, raw, f0, nf):
    """`fh._packed_units` with the number of unit sets per frame (1 unless
    the reader says otherwise: GSB frames are several sets)."""
    units = fh._packed_units(raw, f0, nf)
    return units if len(units) == 6 else tuple(units) + (1,)


def _int8(fh):
    """Whether ``fh`` holds 8-bit two's-complement samples (GUPPI, DADA,
    GSB phased): 8 bits and no level table of its own."""
    return (fh.bps == 8 and getattr(fh, '_codec', None) is None
            and getattr(fh, '_levels', None) is None)


def state_levels(fh):
    """float32 level of every code of ``fh``'s payloads (the decode table;
    for 8-bit two's-complement data the int8 value of every byte)."""
    if _int8(fh):
        return np.arange(256, dtype=np.uint8).view(np.int8).astype(np.float32)
    codec = getattr(fh, '_codec', None)
    lv = codec[1] if codec is not None else getattr(fh, '_levels', None)
    if lv is None:
        raise TypeError('{} has no level table'.format(type(fh).__name__))
    return np.asarray(lv, np.float32)


def _sample_view(fh, table):
    """Per-unit table ``(nbin, nthread, nelem, k)`` of an 8-bit
    two's-complement reader -> ``(nbin,) + sample shape [+ (2,) for complex
    data] + (k,)`` (numpy array or torch tensor)."""
    nbin = table.shape[0]
    view = getattr(fh, '_unit_table_view', None)
    if view is not None:                           # GSB: (pol, chan, parts)
        m = view(table)
        if getattr(fh, 'squeeze', False):
            keep = tuple(d for d in m.shape[1:1 + len(fh._unsliced_shape)]
                         if d > 1)
            m = m.reshape((nbin,) + keep
                          + tuple(m.shape[1 + len(fh._unsliced_shape):]))
        return m
    h0 = fh.header0
    ib = 2 if fh.complex_data else 1
    # (thread = channel, elem = (pol, part)) or (elem = (chan, pol, part))
    m = table.reshape(nbin, h0.nchan, h0.npol, ib, table.shape[-1])
    m = m.swapaxes(1, 2)                           # -> (nbin, npol, nchan, ..)
    if ib == 1:
        m = m[:, :, :, 0]
    if getattr(fh, 'squeeze', False):
        m = m.reshape((nbin,) + tuple(d for d in m.shape[1:3] if d > 1)
                      + tuple(m.shape[3:]))
    return m


def state_counts(fh, samples_per_bin=None, count=None, device_output=False):
    """Occurrences of every code in the next ``count`` samples of ``fh``.

    Returns an int64 array ``(nbin,) + sample shape [+ (2,) for complex
    data] + (2**bps,)``; 8-bit data are counted by the stored byte (index =
    byte value, levels from `state_levels`).  For VDIF the sample shape is
    ``(nthread, nchan)``
    with the threads the reader decodes (its thread subset; unit dimensions
    dropped if the reader squeezes), for Mark 5B and Mark 4 ``(nchan,)``
    (Mark 4: codes indexed ``2 * sign + magnitude`` like its level table,
    counted from the track words; the header steps that open every frame are
    not samples and are left out); for GUPPI, DADA and GSB phased the
    sample shape `moments` returns, and by default the whole frames only, as
    there (GUPPI's overlap samples are left out).  Bin ``b`` covers samples
    ``[b, b + 1) *
    samples_per_bin`` from the current sample pointer (default: one bin);
    frames marked invalid are skipped.  The sample pointer advances by
    ``count``.  The packed frames go host -> HBM once; nothing else moves but
    the counts (``device_output=True`` leaves even those on the GPU).
    """
    int8 = _int8(fh)
    if int8:
        count = _whole_frames(fh, count)
    frame0, nframe, frames_per_bin = _frame_range(fh, count, samples_per_bin)
    nbin = -(-nframe // frames_per_bin)
    state = {}

    own = getattr(fh, '_count_states', None)     # Mark 4: track words

    def consume(raw, f0, nf):
        if own is not None:
            if 'counts' not in state:
                nchan = fh._unsliced_shape[-1]
                state['geom'] = (1, nchan, 2)
                state['counts'] = kernels.zeros((nbin, nchan, 4), torch.int64,
                                                raw.device)
            own(raw, f0, nf, state['counts'], f0 - frame0, frames_per_bin)
            return
        uo, nthread, payload_nbytes, bps, nelem, per = _units(fh, raw, f0, nf)
        if 'counts' not in state:
            state['geom'] = (nthread, nelem, bps)
            state['counts'] = kernels.zeros(
                (nbin, nthread, nelem, 1 << bps), torch.int64, raw.device)
        if bps == 8:
            kernels.byte_counts(raw, uo, nf * per, nthread, payload_nbytes,
                                nelem, state['counts'],
                                set_origin=(f0 - frame0) * per,
                                sets_per_bin=frames_per_bin * per)
        else:
            kernels.state_counts(raw, uo, nf * per, nthread, payload_nbytes,
                                 bps, nelem, state['counts'],
                                 set_origin=(f0 - frame0) * per,
                                 sets_per_bin=frames_per_bin * per)

    fh._for_each_packed_chunk(frame0, nframe, consume)
    check = getattr(fh, '_new_inconsistencies', None)
    if check is not None and getattr(fh, '_index', None) is None and check():
        raise OSError('stream is not a regular sequence of frames; read() '
                      'it once (which indexes it) before counting states.')
    fh.seek(fh.tell() + nframe * fh.samples_per_frame)
    counts = state['counts']
    if int8:
        counts = _sample_view(fh, counts if device_output
                              else counts.cpu().numpy())
        return counts
    nthread, nelem, bps = state['geom']
    shape = tuple(fh._unsliced_shape)
    if getattr(fh, '_decode_ids', None) is not None and len(shape) == 2:
        shape = (nthread, shape[1])
    if getattr(fh, 'squeeze', False):
        shape = tuple(d for d in shape if d > 1)
    if fh.complex_data:
        shape = shape + (2,)
    counts = counts.view((nbin,) + shape + (1 << bps,))
    return counts if device_output else counts.cpu().numpy()


def moments(fh, samples_per_bin=None, count=None):
    """Count, sum and sum of squares of the next ``count`` samples of a
    reader of 8-bit two's-complement data (GUPPI, GSB, DADA), per integration bin and
    sample element, straight from the packed bytes (exact integers).

    Returns three int64 arrays ``(n, total, total_of_squares)`` of shape
    ``(nbin,) + sample shape [+ (2,) for complex data]``.  Bins cover whole
    frames from the current sample pointer; GUPPI's overlap samples, which
    repeat in the next frame, are left out, and so is the overlap that ends
    the file.  The sample pointer advances by ``count``."""
    frame0, nframe, frames_per_bin = _frame_range(fh, _whole_frames(fh, count),
                                                  samples_per_bin)
    nbin = -(-nframe // frames_per_bin)
    state = {}

    def consume(raw, f0, nf):
        uo, nthread, payload_nbytes, bps, nelem, per = _units(fh, raw, f0, nf)
        if bps != 8:
            raise TypeError('moments are for 8-bit data; use state_counts')
        if 'm' not in state:
            state['geom'] = (nthread, nelem)
            state['m'] = kernels.zeros((nbin, nthread, nelem, 3), torch.int64,
                                       raw.device)
        kernels.int8_moments(raw, uo, nf * per, nthread, payload_nbytes,
                             nelem, state['m'],
                             set_origin=(f0 - frame0) * per,
                             sets_per_bin=frames_per_bin * per)

    fh._for_each_packed_chunk(frame0, nframe, consume)
    fh.seek(fh.tell() + nframe * fh.samples_per_frame)
    m = _sample_view(fh, state['m'].cpu().numpy())
    return m[..., 0], m[..., 1], m[..., 2]


def _whole_frames(fh, count):
    """Default count for formats whose stream ends in an overlap: all whole
    frames from the sample pointer."""
    if count is not None:
        return count
    spf = fh.samples_per_frame
    whole = min(fh._nframe * spf, fh.shape[0] // spf * spf)   # DADA: the last
    return whole - fh.tell()                                  # may be short


def integrated_power(fh, samples_per_bin=None, count=None, average=True):
    """Power per integration bin: ``Integrate(Square(fh), samples_per_bin)``
    of the baseband-tasks vocabulary, computed from `state_counts` (float64:
    ``sum_c counts[c] * level[c]**2``; for complex data re**2 + im**2).
    With ``average`` the mean over the valid samples of the bin (NaN for a
    bin without valid samples), else the sum."""
    if _int8(fh):
        # 8-bit two's complement: from the moments
        n, _, sq = moments(fh, samples_per_bin, count)
        total = sq.astype(np.float64)
        if fh.complex_data:
            total, n = total.sum(-1), n[..., 0]
        if not average:
            return total
        with np.errstate(invalid='ignore', divide='ignore'):
            return total / n
    lv = state_levels(fh).astype(np.float64)
    counts = state_counts(fh, samples_per_bin, count)
    total = (counts * lv ** 2).sum(-1)
    nvalid = counts.sum(-1)
    if fh.complex_data:
        total = total.sum(-1)
        nvalid = nvalid[..., 0]
    if not average:
        return total
    with np.errstate(invalid='ignore', divide='ignore'):
        return total / nvalid
