"""Subset reads: decode + gather against the selective decoders on the GPU.

    python tools/bench_subset.py [--gib 1] [--seconds 2]

Device-resident chunks of --gib packed bytes (well above the 126 MB L2),
unit tables built once, so only the decode work is timed.  Two legs per
shape, alternating in blocks of about a quarter second with CUDA events
until each has --seconds:
  gather  the full-width decoder into a scratch buffer, then the torch index
          a reader applied to the decoded rows before (`_finish`)
  select  bb_decode_select_bitfield / bb_decode_select_int8 straight into the
          selected width
Both outputs are compared bitwise in the same run.  The C4 shapes lie on
both sides of the readers' choice to decode whole rows and gather for
int8 subsets of at least 7/8 of the row (`_gather_fraction`).  Reports each leg's time,
output Gsamples/s (selected components per second) and the algorithmic
TB/s: (32-byte packed sectors the selection needs + output bytes) / time.
bb_probe_copy (read + write of 1 GiB) is the ceiling.  Then a public-API
leg: a device read of a C4 GUPPI single-channel subset from a pinned
HostBuffer against the same read without a subset, with its rate and peak
device memory.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(
    __file__))))
import baseband_b200 as bb  # noqa: E402
from baseband_b200 import kernels, levels, synthetic  # noqa: E402
from baseband_b200.base.memory import HostBuffer  # noqa: E402

DEV = torch.device('cuda:0')


def card():
    name = torch.cuda.get_device_name(DEV)
    try:
        power = subprocess.run(
            ['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader',
             '-i', '0'], capture_output=True, text=True, timeout=30
        ).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def timed(legs, seconds):
    """Alternate the callables of ``legs`` in ~0.25 s blocks; seconds per
    call of each."""
    per = {}
    for name, fn in legs.items():
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        per[name] = max(1, int(0.25 / max(time.perf_counter() - t0, 1e-6)))
    total = {k: 0. for k in legs}
    calls = {k: 0 for k in legs}
    while min(total.values()) < seconds:
        for name, fn in legs.items():
            a, b = torch.cuda.Event(True), torch.cuda.Event(True)
            a.record()
            for _ in range(per[name]):
                fn()
            b.record()
            b.synchronize()
            total[name] += a.elapsed_time(b) / 1e3
            calls[name] += per[name]
    return {k: total[k] / calls[k] for k in legs}


def sectors(positions, unit_nbytes, nunit):
    """32-byte sectors of ``nunit`` units holding the byte ``positions`` of
    one unit."""
    per = np.unique(np.asarray(positions, np.int64) // 32).size
    return per * 32 * nunit


def bitfield_shape(label, gib, nthread, nelem, bps, payload, codec, lv, sel,
                   dtype=torch.float32, complex_data=False):
    nunit_total = int(gib * (1 << 30)) // payload
    nset = nunit_total // nthread
    spf = payload * 8 // (bps * nelem)
    g = torch.Generator(device=DEV).manual_seed(7)
    raw = torch.randint(0, 256, (nset * nthread * payload,), dtype=torch.uint8,
                        device=DEV, generator=g)
    uo = torch.arange(nset * nthread, dtype=torch.int64, device=DEV) * payload
    nsample = nset * spf
    width = nthread * nelem
    sel = np.asarray(sel, np.int32)
    sel_d = torch.from_numpy(sel).to(DEV)
    idx = torch.from_numpy(sel.astype(np.int64)).to(DEV)
    scratch = torch.empty(nsample * width, dtype=dtype, device=DEV)
    out = torch.empty(nsample * sel.size, dtype=dtype, device=DEV)
    args = (raw, uo, nset, nthread, payload, bps, nelem, complex_data, codec,
            lv, 0., 0, nsample)
    res = {}

    def gather():
        kernels.decode_bitfield(*args, out=scratch)
        res['gather'] = scratch.view(nsample, width)[:, idx]

    def select():
        kernels.decode_select_bitfield(*args, sel_d, out)
    slot, e = np.divmod(sel, nelem)
    t = np.arange(spf, dtype=np.int64)[:, None]
    need = sum(sectors((t * nelem + e[slot == k]) * bps // 8, payload,
                       nset) for k in np.unique(slot))
    return report(label, gather, select, res, out, nsample * sel.size,
                  need, dtype)


def guppi_shape(label, gib, sel_comp, nchan=512, npol=2, spf=4096):
    ib = 2
    unit = nchan * spf * npol * ib
    nunit = max(1, int(gib * (1 << 30)) // unit)
    g = torch.Generator(device=DEV).manual_seed(8)
    raw = torch.randint(0, 256, (nunit * unit,), dtype=torch.uint8,
                        device=DEV, generator=g)
    uo = torch.arange(nunit, dtype=torch.int64, device=DEV) * unit
    begin = torch.zeros(nunit, dtype=torch.int64, device=DEV)
    end = torch.full((nunit,), spf, dtype=torch.int64, device=DEV)
    first = torch.arange(nunit, dtype=torch.int64, device=DEV) * spf
    sel = np.asarray(sel_comp, np.int64)
    pol, rest = np.divmod(sel, nchan * ib)
    chan, part = np.divmod(rest, ib)
    off = chan * spf * npol * ib + pol * ib + part
    off_d = torch.from_numpy(off.astype(np.int32)).to(DEV)
    idx = torch.from_numpy(sel).to(DEV)
    width = npol * nchan * ib
    nsample = nunit * spf
    scratch = torch.empty(nsample * width, device=DEV)
    out = torch.empty(nsample * sel.size, device=DEV)
    res = {}

    def gather():
        kernels.decode_int8_transposed(raw, uo, nunit, nchan, spf * npol, ib,
                                       begin * npol, end * npol,
                                       first * npol, scratch)
        res['gather'] = scratch.view(nsample, width)[:, idx]

    def select():
        kernels.decode_select_int8(raw, uo, nunit, spf, spf, 0, npol * ib,
                                   off_d, begin, end, first, out)
    t = np.arange(spf, dtype=np.int64)[:, None]
    need = sectors(t * npol * ib + off, unit, nunit)
    return report(label, gather, select, res, out, nsample * sel.size, need,
                  torch.float32)


def report(label, gather, select, res, out, nout, need, dtype):
    times = timed({'gather': gather, 'select': select}, ARGS.seconds)
    gather()
    select()
    torch.cuda.synchronize()
    a = res['gather'].reshape(-1)
    bits = torch.int32 if dtype == torch.float32 else torch.int16
    equal = bool(torch.equal(a.contiguous().view(bits), out.view(bits)))
    nbytes = need + nout * out.element_size()
    row = {'shape': label, 'gather_ms': times['gather'] * 1e3,
           'select_ms': times['select'] * 1e3,
           'speedup': times['gather'] / times['select'],
           'select_gsamples_s': nout / times['select'] / 1e9,
           'select_tb_s': nbytes / times['select'] / 1e12,
           'gather_gsamples_s': nout / times['gather'] / 1e9,
           'outputs_equal': equal}
    print('%-44s gather %8.3f ms  select %8.3f ms  x%5.2f  %6.2f Gsamp/s  '
          '%5.2f TB/s  %s' % (label, row['gather_ms'], row['select_ms'],
                              row['speedup'], row['select_gsamples_s'],
                              row['select_tb_s'],
                              'equal' if equal else 'DIFFER'), flush=True)
    del res['gather']
    torch.cuda.empty_cache()
    return row


def api_leg():
    raw, _ = synthetic.guppi_stream(32, nchan=512, npol=2,
                                    samples_per_frame=4096, overlap=0, seed=5)
    rows = {}
    for label, kw in (('subset (0, 7)', {'subset': (0, 7)}), ('full', {})):
        best, peak = None, 0
        for _ in range(3):
            src = HostBuffer(raw)             # closed with its reader
            with bb.guppi.open(src, 'rs', device=DEV, **kw) as fh:
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                t0 = time.perf_counter()
                data = fh.read()
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                peak = torch.cuda.max_memory_allocated() - base
                del data
            best = dt if best is None else min(best, dt)
        rows[label] = {'seconds': best, 'packed_gb_s': raw.size / best / 1e9,
                       'peak_device_mib': peak / 2**20}
        print('api guppi C4 device read, %-14s %7.3f s  %6.2f GB/s packed  '
              'peak %8.1f MiB' % (label, best, raw.size / best / 1e9,
                                  peak / 2**20), flush=True)
    return rows


def main():
    global ARGS
    p = argparse.ArgumentParser()
    p.add_argument('--gib', type=float, default=1.0)
    p.add_argument('--seconds', type=float, default=2.0)
    ARGS = p.parse_args()
    name, power = card()
    print('card: %s, power limit %s' % (name, power), flush=True)
    n = int(ARGS.gib * (1 << 30))
    a = torch.empty(n, dtype=torch.uint8, device=DEV)
    b = torch.empty(n, dtype=torch.uint8, device=DEV)
    t = timed({'copy': lambda: kernels.probe_copy(b, a)}, ARGS.seconds)
    copy_tb_s = 2 * n / t['copy'] / 1e12
    print('bb_probe_copy ceiling: %.2f TB/s (read + write)' % copy_tb_s)
    del a, b
    rows = []
    m5b = levels.mark5b(2)
    for label, sel, dtype in (
            ('C5 mark5b 16ch 2bit: 2 of 16', [3, 9], torch.float32),
            ('C5 mark5b 16ch 2bit: 15 of 16',
             [i for i in range(16) if i != 4], torch.float32),
            ('C5 mark5b 16ch 2bit: 2 of 16, float16', [3, 9],
             torch.float16)):
        rows.append(bitfield_shape(label, ARGS.gib, 1, 16, 2, 10000,
                                   kernels.CODEC_LEVELS, m5b, sel, dtype))
    rows.append(bitfield_shape(
        '8-bit time-first 2048 comp: 4 of 2048', ARGS.gib, 1, 2048, 8,
        64 << 20, kernels.CODEC_SINT, None, [0, 1, 1024, 1025]))
    rows.append(bitfield_shape(
        'VDIF 4 thr x 8 ch 2bit: ch 3 of each', ARGS.gib, 4, 8, 2, 8000,
        kernels.CODEC_LEVELS, levels.offset_binary(2), [3, 11, 19, 27]))
    comp = np.arange(2 * 512 * 2)
    pol, chan = comp // 1024, comp % 1024 // 2
    for label, keep in (
            ('C4 guppi: 64 adjacent channels of pol 0',
             (pol == 0) & (chan >= 100) & (chan < 164)),
            ('C4 guppi: one channel, both pols', chan == 7),
            ('C4 guppi: all but one channel', chan != 7)):
        rows.append(guppi_shape(label, ARGS.gib, comp[keep]))
    api = api_leg()
    print(json.dumps({'card': name, 'power_limit': power,
                      'probe_copy_tb_s': copy_tb_s, 'shapes': rows,
                      'api': api}))


if __name__ == '__main__':
    main()
