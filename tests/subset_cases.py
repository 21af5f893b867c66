"""Subset reads decoded by the selective kernels: the kernels against numpy
restatements on seeded random geometries, and every format's reader with a
``subset`` against the same reader without one, indexed afterwards, bit for
bit.  Shared by tests/test_host_subset.py (CPU emulation backend, ``dev =
'cpu'``) and tests/test_gpu_subset.py (B200)."""
import pickle

import numpy as np
import pytest
import torch

from baseband_b200 import kernels, levels as _levels
import reduced_cases

OUT_TYPES = (torch.float32, torch.float16, torch.bfloat16)


def same(got, want):
    """Bitwise equality of two results (numpy or torch, any device): dtype,
    shape and every bit, -0.0 included; NaN by position (a reduced type's
    NaN payload is not specified)."""
    g, w = reduced_cases.as_pairs(got), reduced_cases.as_pairs(want)
    assert g.dtype == w.dtype, (g.dtype, w.dtype)
    assert tuple(g.shape) == tuple(w.shape), (g.shape, w.shape)
    gn, wn = torch.isnan(g.float()), torch.isnan(w.float())
    assert torch.equal(gn, wn), 'NaN positions differ'
    bits = {4: torch.int32, 2: torch.int16}[g.element_size()]
    gb = g.contiguous().view(bits)[~gn]
    wb = w.contiguous().view(bits)[~wn]
    if not torch.equal(gb, wb):
        bad = (gb != wb).nonzero()[:5].tolist()
        raise AssertionError('{} of {} values differ, e.g. at {}'.format(
            int((gb != wb).sum()), gb.numel(), bad))


# ------------------------------------------------------------ kernel level
def selections(rng, width):
    """Selections of a row of ``width`` components: a single one, runs,
    strided runs, repeats, reversed, near-full, odd lengths."""
    out = [[int(rng.integers(width))], list(range(width))[::-1],
           list(range(0, width, 3)) or [0],
           [i for i in range(width) if i != width // 2] or [0],
           list(rng.integers(0, width, 5)),
           list(range(min(width, 64))) * 2]
    a = int(rng.integers(width))
    out.append(list(range(a, min(width, a + 3))))
    return [np.asarray(s, np.int32) for s in out]


def oracle_bitfield(raw, uo, nset, nthread, payload_nbytes, bps, nelem,
                    complex_data, lv, fill, sample_start, nsample, sel):
    """Rows of bb_decode_bitfield restated with numpy, then the columns
    ``sel``: float32 (nsample, len(sel))."""
    spf = payload_nbytes * 8 // (bps * nelem)
    full = np.empty((nset, spf, nthread, nelem), np.float32)
    shifts = np.arange(0, 32, bps, dtype=np.uint32)
    for s in range(nset):
        for k in range(nthread):
            off = int(uo[s * nthread + k])
            if off < 0:
                full[s, :, k] = np.float32(fill)
                if complex_data:
                    full[s, :, k, 1::2] = 0.
                continue
            w = raw[off:off + payload_nbytes].view('<u4')
            codes = ((w[:, None] >> shifts) & ((1 << bps) - 1)).reshape(
                spf, nelem).astype(np.int64)
            if lv is None:
                codes = np.where(codes >= 1 << (bps - 1), codes - (1 << bps),
                                 codes)
                full[s, :, k] = codes
            else:
                full[s, :, k] = lv[codes]
    rows = full.reshape(nset * spf, nthread * nelem)
    return rows[sample_start:sample_start + nsample][:, sel]


def bitfield_cases(n=24, seed=11):
    """Random geometries: bps 1/2/4/8, 1-64 threads, nelem 1-2048, real and
    complex, invalid units, reads cutting units, every codec."""
    rng = np.random.default_rng(seed)
    cases = []
    for i in range(n):
        bps = (1, 2, 4, 8)[i % 4]
        nthread = int(rng.choice([1, 2, 3, 4, 8, 16, 64]))
        complex_data = bool(i % 3 == 1)
        nelem = int(rng.choice([1, 2, 3, 4, 8, 16, 160, 2048]))
        if complex_data:
            nelem = 2 * max(1, nelem // 2)
        # whole samples in whole words, a few samples per unit
        per = np.lcm(32, bps * nelem) // (bps * nelem)
        spf = int(per * rng.integers(1, max(2, 64 // per + 1)))
        while spf * nthread * nelem > 20000 and spf > per:
            spf -= per
        payload_nbytes = spf * bps * nelem // 8
        nset = int(rng.integers(1, 5))
        if bps in (4, 8) and i % 5 == 2:
            codec, lv = kernels.CODEC_SINT, None
        elif bps == 8 and i % 2:
            codec, lv = kernels.CODEC_LEVELS, _levels.offset_binary(8)
        else:
            codec = kernels.CODEC_LEVELS
            lv = rng.normal(size=1 << bps).astype(np.float32)
            lv[0] = -0.
        start = int(rng.integers(0, spf))
        nsample = int(rng.integers(1, nset * spf - start + 1))
        cases.append(dict(bps=bps, nthread=nthread, nelem=nelem,
                          complex_data=complex_data, spf=spf,
                          payload_nbytes=payload_nbytes, nset=nset,
                          codec=codec, levels=lv, start=start,
                          nsample=nsample, seed=int(rng.integers(1 << 30)),
                          fill=float(rng.choice([0., -0., 7.5, np.nan]))))
    return cases


def check_bitfield(case, dev):
    c = case
    rng = np.random.default_rng(c['seed'])
    nunit = c['nset'] * c['nthread']
    raw = rng.integers(0, 256, nunit * c['payload_nbytes'] + 64, np.uint8)
    uo = (np.arange(nunit, dtype=np.int64) * c['payload_nbytes'] + 16)
    uo[rng.random(nunit) < 0.2] = -1
    width = c['nthread'] * c['nelem']
    for k, sel in enumerate(selections(rng, width)):
        want = oracle_bitfield(raw, uo, c['nset'], c['nthread'],
                               c['payload_nbytes'], c['bps'], c['nelem'],
                               c['complex_data'], c['levels'], c['fill'],
                               c['start'], c['nsample'], sel)
        dtype = OUT_TYPES[k % 3]
        lead = k % 4                       # output off the 4-element grid
        n = want.size
        buf = torch.full((n + lead + 3,), 99., dtype=dtype, device=dev)
        out = buf[lead:lead + n]
        kernels.decode_select_bitfield(
            torch.from_numpy(raw).to(dev), torch.from_numpy(uo).to(dev),
            c['nset'], c['nthread'], c['payload_nbytes'], c['bps'],
            c['nelem'], c['complex_data'], c['codec'], c['levels'],
            c['fill'], c['start'], c['nsample'],
            torch.from_numpy(sel).to(dev), out)
        same(out, torch.from_numpy(want).reshape(-1).to(dtype))
        assert bool((buf[:lead] == 99).all() and (buf[lead + n:] == 99).all())


def check_bitfield_launch_split(dev):
    """A selection wider than the shared-memory table, and an entry outside
    the row (written as NaN)."""
    rng = np.random.default_rng(3)
    nthread, nelem, spf, nset = 3, 1000, 32, 2
    payload = spf * nelem * 2 // 8
    raw = rng.integers(0, 256, nset * nthread * payload, np.uint8)
    uo = np.arange(nset * nthread, dtype=np.int64) * payload
    sel = rng.integers(0, nthread * nelem, 2500).astype(np.int32)
    lv = _levels.offset_binary(2)
    want = oracle_bitfield(raw, uo, nset, nthread, payload, 2, nelem, False,
                           lv, 0., 5, 50, sel)
    out = torch.empty(want.size, device=dev)
    args = (torch.from_numpy(raw).to(dev), torch.from_numpy(uo).to(dev),
            nset, nthread, payload, 2, nelem, False, kernels.CODEC_LEVELS, lv,
            0., 5, 50)
    kernels.decode_select_bitfield(*args, torch.from_numpy(sel).to(dev), out)
    same(out, torch.from_numpy(want).reshape(-1))
    bad = np.array([0, nthread * nelem, -1, 1], np.int32)
    out = torch.empty(50 * 4, device=dev)
    kernels.decode_select_bitfield(*args, torch.from_numpy(bad).to(dev), out)
    got = out.cpu().view(50, 4)
    assert torch.isnan(got[:, 1:3]).all()
    ok = oracle_bitfield(raw, uo, nset, nthread, payload, 2, nelem, False,
                         lv, 0., 5, 50, bad[[0, 3]])
    same(got[:, [0, 3]].contiguous(), torch.from_numpy(ok))


def oracle_int8(raw, uo, heap, heap_stride, t_stride, off, t_begin, t_end,
                out_t0, nrow):
    out = np.full((nrow, off.size), np.nan, np.float32)
    vals = raw.view(np.int8)
    for u in range(len(uo)):
        for k, t in enumerate(range(t_begin[u], t_end[u])):
            at = (uo[u] + t // heap * heap_stride + t % heap * t_stride
                  + off.astype(np.int64))
            out[out_t0[u] + k] = vals[at]
    return out


def int8_cases():
    """GUPPI channels-first and time-first frames with overlap windows, and
    MKBF heaps, each with several selections."""
    cases = []
    for layout in ('chan_first', 'time_first', 'mkbf'):
        for nchan, npol, ib in ((5, 2, 2), (8, 1, 1), (64, 2, 2)):
            cases.append((layout, nchan, npol, ib))
    return cases


def check_int8(case, dev):
    layout, nchan, npol, ib = case
    rng = np.random.default_rng(nchan * 7 + npol)
    width = npol * nchan * ib
    comp = np.arange(width)
    pol, rest = np.divmod(comp, nchan * ib)
    chan, part = np.divmod(rest, ib)
    if layout == 'mkbf':
        heap, nsample, nunit = 256, 256 * 3, 1
        heap_stride, t_stride = width * 256, ib
        offs = (pol * nchan + chan) * 256 * ib + part
        t_begin, t_end, out_t0 = [37], [37 + 700], [0]
    else:
        nsample, nunit = 40, 3
        heap, heap_stride = nsample, 0
        if layout == 'chan_first':
            offs, t_stride = chan * nsample * npol * ib + pol * ib + part, \
                npol * ib
        else:
            offs, t_stride = (chan * npol + pol) * ib + part, nchan * npol * ib
        # overlap 6: the first frame from sample 3, the rest from 6 on, the
        # last one cut short
        t_begin, t_end = [3, 6, 6], [40, 40, 25]
        out_t0 = list(np.concatenate([[0], np.cumsum(
            np.subtract(t_end, t_begin))[:-1]]))
    unit_nbytes = nsample * width
    raw = rng.integers(0, 256, nunit * unit_nbytes + 40, np.uint8)
    uo = np.arange(nunit, dtype=np.int64) * unit_nbytes + 8
    nrow = int(np.sum(np.subtract(t_end, t_begin)))
    tables = [torch.tensor(np.asarray(x, np.int64), device=dev)
              for x in (uo, t_begin, t_end, out_t0)]
    for k, sel in enumerate(selections(rng, width)):
        off = offs[sel].astype(np.int32)
        want = oracle_int8(raw, uo, heap, heap_stride, t_stride, off,
                           t_begin, t_end, out_t0, nrow)
        dtype = OUT_TYPES[k % 3]
        lead = (k + 1) % 4
        buf = torch.full((want.size + lead + 2,), 99., dtype=dtype, device=dev)
        out = buf[lead:lead + want.size]
        kernels.decode_select_int8(
            torch.from_numpy(raw).to(dev), tables[0], nunit, nsample, heap,
            heap_stride, t_stride, torch.from_numpy(off).to(dev), tables[1],
            tables[2], tables[3], out)
        same(out, torch.from_numpy(want).reshape(-1).to(dtype))
        assert bool((buf[:lead] == 99).all()
                    and (buf[lead + want.size:] == 99).all())


# ------------------------------------------------------------ public API
def subsets(shape):
    """The subsets to try on samples of ``shape`` (each as far as the
    reader accepts it)."""
    n0 = shape[0] if shape else 1
    return [0, -1, slice(1, None, 3), [3, 1, 3], np.arange(n0) % 2 == 0,
            (0, slice(100, 200)), (0, slice(1, None, 2)), ([0, 1], [2, 3]),
            np.array([1, 0]), (slice(None), [-1, 0])]


def _opened(opener, **kw):
    try:
        return opener(**kw)
    except (IndexError, AssertionError, TypeError, ValueError):
        return None                    # a subset this reader refuses


def check_stream(name, dev):
    """Every subset on stream ``name``, squeeze on and off: host and device
    output, partial reads, float16, against the full read indexed."""
    make, has_fill, reads = reduced_cases.STREAMS[name]
    opener = make()
    fill = {'fill_value': -0.} if has_fill else {}
    ntried = 0
    for squeeze in (True, False, None):
        kw = dict(fill) if squeeze is None else dict(fill, squeeze=squeeze)
        ref = _opened(opener, **kw)
        if ref is None or (squeeze is None and ntried):
            continue            # squeeze given, or a reader that fixes it
        with ref:
            full = ref.read()
            shape = ref.sample_shape
        for subset in subsets(tuple(shape)):
            fh = _opened(opener, subset=subset, **kw)
            if fh is None:
                continue
            index = (slice(None),) + (subset if isinstance(subset, tuple)
                                      else (subset,))
            # (an irregular stream indexed for fewer threads may end sooner)
            spans = reads(fh.shape[0])
            with fh:
                try:
                    got = fh.read(spans[0][1])
                except RuntimeError:
                    # a subset the reader shapes unlike numpy is refused
                    # when read, as it was before
                    continue
                ntried += 1
                same(got, full[:spans[0][1]][index])
                for start, count in spans[1:]:
                    fh.seek(start)
                    same(fh.read(count), full[start:start + count][index])
            with opener(subset=subset, device=dev, **kw) as fh:
                for start, count in spans:
                    fh.seek(start)
                    got = fh.read(count)
                    assert isinstance(got, torch.Tensor)
                    same(got, full[start:start + count][index])
            with opener(subset=subset, device=dev, dtype='float16',
                        **kw) as fh:
                start, count = spans[1]
                fh.seek(start)
                reduced_cases.assert_reduced(
                    fh.read(count), full[start:start + count][index],
                    torch.float16)
    assert ntried >= 3


def check_ways_of_reading(dev, name='vdif_synth16', subset=(slice(2, 9, 3),)):
    """out= of every kind, on_device, small cached reads, many chunks and
    pickling, all with a subset."""
    make, _, _ = reduced_cases.STREAMS[name]
    opener = make()
    with opener() as ref:
        full = ref.read()
    index = (slice(None),) + subset
    want = full[index]
    with opener(subset=subset) as fh:
        assert fh.shape == want.shape
        same(fh.read(), want)                              # many chunks
        fh.seek(5)
        same(fh.read(3), want[5:8])                        # small, cached
        out = np.empty(want[8:4008].shape, np.float32)
        assert fh.read(out=out) is out
        same(out, want[8:4008])
        clone = pickle.loads(pickle.dumps(fh))
        same(clone.read(100), want[4008:4108])
        clone.close()
        t = torch.empty(tuple(want[:777].shape))
        fh.seek(1)
        assert fh.read(out=t) is t
        same(t, want[1:778])
    with opener(subset=subset, device=dev) as fh:
        seen = []
        fh.seek(3)
        got = fh.read(60001, on_device=lambda p: seen.append(p.clone()))
        same(got, want[3:60004])
        same(torch.cat(seen), want[3:60004])
        for lead in (0, 1, 3):                 # device out=, any alignment
            buf = torch.empty(want[:1000].size + lead, device=dev)
            out = buf[lead:].view(want[:1000].shape)
            fh.seek(0)
            assert fh.read(out=out) is out
            same(out, want[:1000])
        out = torch.empty(want[:1000].shape, device=dev).t().contiguous().t()
        fh.seek(0)
        assert fh.read(out=out) is out                    # non-contiguous
        same(out, want[:1000])
    for dtype in (torch.float16, torch.bfloat16):
        with opener(subset=subset, device=dev) as fh:
            out = torch.empty(want[:999].shape, dtype=dtype, device=dev)
            assert fh.read(out=out) is out
            reduced_cases.assert_reduced(out, want[:999], dtype)
