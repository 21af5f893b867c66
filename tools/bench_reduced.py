"""float32 vs float16 / bfloat16 decoder output on the GPU.

    python tools/bench_reduced.py [--gib 1] [--seconds 2] [--dump DIR]

Device-resident decode of the named shapes, the unit tables built once so
that only the decode kernel is timed:
  C1  VDIF, sample.vdif geometry: 8 threads, 2 bit, 5000-byte payloads
  C2  VDIF, 16 threads, 2 bit, 8000-byte payloads (the headline shape)
  C3  Mark 4, 64 tracks, fan-out 4, 8 channels (header rows -> fill)
  C4  GUPPI, 512 channels, 2 pol, 8-bit complex, channels first, overlap
  C5  Mark 5B, 16 channels, 2 bit, 1 % invalid frames (fill)
Each shape gets --gib of packed input (well beyond the 126 MB L2), is warmed
up, and is timed with CUDA events in blocks of about a quarter second,
float32 / float16 / bfloat16 blocks alternating, until every leg has
--seconds.  bb_probe_copy is timed in the same run.  Then a host-output read
of C2 through the public API (``read(out=pinned)`` from a HostBuffer) at
float32 and float16, alternating.

Reports Gsamples/s, the algorithmic TB/s (packed bytes read + output bytes
written), the ratio to float32, and whether every reduced output equals the
float32 output converted by torch (NaN by position); the card's name and
power limit are read in the same run.  --dump DIR writes the first 2^18
values of every output of every shape (fixed seeds; the 16-bit types as
their uint16 bit patterns) as .npy for offline comparison.
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
from baseband_b200 import kernels, levels, synthetic  # noqa: E402

TYPES = (torch.float32, torch.float16, torch.bfloat16)
NAMES = {torch.float32: 'float32', torch.float16: 'float16',
         torch.bfloat16: 'bfloat16'}


def card():
    info = {'name': torch.cuda.get_device_name()}
    try:
        q = subprocess.run(
            ['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm',
             '--format=csv,noheader', '-i',
             str(torch.cuda.current_device())],
            capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        info['power_limit_and_max_sm_clock'] = 'unknown ({})'.format(exc)
    return info


def exact(got, want32):
    """``got`` == ``want32.to(got.dtype)`` bitwise, NaN by position."""
    g = got.reshape(-1)
    exp = want32.reshape(-1).to(g.dtype)
    gn, en = torch.isnan(g), torch.isnan(exp)
    if not torch.equal(gn, en):
        return False
    return torch.equal(g.view(torch.int16)[~gn], exp.view(torch.int16)[~en])


def time_legs(fns, seconds):
    """fns: {key: callable}.  Alternating blocks of CUDA-event-timed calls
    until every key has ``seconds``; returns {key: seconds per call}."""
    for fn in fns.values():                      # warm-up
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    per_block = {}
    for k, fn in fns.items():                    # calls per ~0.25 s block
        a, b = (torch.cuda.Event(enable_timing=True) for _ in range(2))
        a.record()
        fn()
        b.record()
        b.synchronize()
        per_block[k] = max(1, int(0.25 / max(a.elapsed_time(b) * 1e-3,
                                             1e-6)))
    total = {k: 0.0 for k in fns}
    calls = {k: 0 for k in fns}
    while min(total.values()) < seconds:
        for k, fn in fns.items():
            a, b = (torch.cuda.Event(enable_timing=True) for _ in range(2))
            a.record()
            for _ in range(per_block[k]):
                fn()
            b.record()
            b.synchronize()
            total[k] += a.elapsed_time(b) * 1e-3
            calls[k] += per_block[k]
    return {k: total[k] / calls[k] for k in fns}, total


def shapes(nbytes, dev):
    """name -> (packed bytes, decode(out), output numel)."""
    out = {}
    # C1 / C2: VDIF, all frames valid
    for name, nthread, payload in (('C1_vdif_8thread_2bit', 8, 5000),
                                   ('C2_vdif_16thread_2bit', 16, 8000)):
        frame = payload + 32
        nset = nbytes // (nthread * frame)
        raw = synthetic.vdif_stream_device(nset, nthread, payload, dev,
                                           seed=synthetic.VDIF_SEED)
        uo = (torch.arange(nset * nthread, dtype=torch.int64, device=dev)
              * frame + 32)
        lv = levels.offset_binary(2)
        n = nset * payload * 4 * nthread

        def dec(o, raw=raw, uo=uo, nset=nset, nthread=nthread,
                payload=payload, lv=lv):
            kernels.decode_bitfield(raw, uo, nset, nthread, payload, 2, 1,
                                    False, kernels.CODEC_LEVELS, lv, out=o)
        out[name] = (raw.numel(), dec, n)
    # C3: Mark 4
    nframe = nbytes // 160000
    raw4 = synthetic.mark4_stream_device(nframe, dev,
                                         seed=synthetic.MARK4_SEED)
    _, uo4 = kernels.mark4_scan(raw4, nframe, 64)
    lv4 = levels.sign_magnitude()

    def c3(o):
        kernels.mark4_decode(raw4, uo4, nframe, 8, 4, False, lv4, out=o)
    out['C3_mark4_64track_fanout4'] = (raw4.numel(), c3, nframe * 80000 * 8)
    # C4: GUPPI channels first, overlap columns skipped
    nchan, npol, spf, ov = 512, 2, 65536, 512
    fbytes = nchan * spf * npol * 2
    nfr = max(1, nbytes // fbytes)
    g = torch.Generator(device=dev).manual_seed(synthetic.GUPPI_SEED)
    rawg = torch.randint(0, 256, (nfr * fbytes,), dtype=torch.uint8,
                         device=dev, generator=g)
    off = torch.arange(nfr, dtype=torch.int64, device=dev) * fbytes
    cb = torch.zeros(nfr, dtype=torch.int64, device=dev)
    ce = torch.full((nfr,), (spf - ov) * npol, dtype=torch.int64, device=dev)
    ce[-1] = spf * npol
    oc0 = torch.cumsum(ce - cb, 0) - (ce - cb)
    ncols = int((ce - cb).sum().item())

    def c4(o):
        kernels.decode_int8_transposed(rawg, off, nfr, nchan, spf * npol, 2,
                                       cb, ce, oc0, o)
    # packed bytes read: the non-overlap input (as bench.py counts them)
    out['C4_guppi_512chan_2pol_int8_complex'] = (ncols * nchan * 2, c4,
                                                 ncols * nchan * 2)
    # C5: Mark 5B with 1 % fill-pattern frames
    nframe5 = nbytes // 10016
    raw5, _ = synthetic.mark5b_stream_device(nframe5, dev,
                                             seed=synthetic.MARK5B_SEED)
    _, uo5 = kernels.mark5b_scan(raw5, nframe5)
    lv5 = levels.mark5b(2)

    def c5(o):
        kernels.decode_bitfield(raw5, uo5, nframe5, 1, 10000, 2, 16, False,
                                kernels.CODEC_LEVELS, lv5, -999.0, out=o)
    out['C5_mark5b_2bit_16chan_1pct_invalid'] = (raw5.numel(), c5,
                                                 nframe5 * 2500 * 16)
    return out


def bench_device(args, dev):
    result = {}
    nbytes = int(args.gib * 2**30)
    for name, (packed, dec, n) in shapes(nbytes, dev).items():
        bufs = {t: torch.empty(n, dtype=t, device=dev) for t in TYPES}
        per_call, total = time_legs(
            {t: (lambda t=t: dec(bufs[t])) for t in TYPES}, args.seconds)
        torch.cuda.synchronize()
        row = {'packed_bytes': packed, 'nsamples': n}
        for t in TYPES:
            s = per_call[t]
            row[NAMES[t]] = {
                'ms_per_call': s * 1e3, 'seconds_timed': total[t],
                'gsamples_s': n / s / 1e9,
                'algo_tb_s': (packed + n * bufs[t].element_size()) / s / 1e12,
                'ratio_to_float32': per_call[torch.float32] / s}
            if t != torch.float32:
                row[NAMES[t]]['exact'] = bool(exact(bufs[t],
                                                    bufs[torch.float32]))
        if args.dump:
            k = min(n, 1 << 18)
            for t in TYPES:
                a = bufs[t][:k].cpu()
                a = a.numpy() if t == torch.float32 else \
                    a.view(torch.int16).numpy().view(np.uint16)
                np.save(os.path.join(args.dump, '{}_{}.npy'.format(
                    name, NAMES[t])), a)
        result[name] = row
        print(json.dumps({name: row}), flush=True)
        del bufs
        torch.cuda.empty_cache()
    # copy ceiling in the same run
    half = 2**30
    a = torch.empty(half // 4, dtype=torch.float32, device=dev)
    b = torch.zeros_like(a)
    per, _ = time_legs({'copy': lambda: kernels.probe_copy(a, b)},
                       min(args.seconds, 1.0))
    result['bb_probe_copy'] = {'tb_s': 2 * half / per['copy'] / 1e12,
                               'bytes_per_call': 2 * half}
    print(json.dumps({'bb_probe_copy': result['bb_probe_copy']}), flush=True)
    return result


def bench_host(args):
    """read(out=pinned) of C2 from a HostBuffer, float32 vs float16."""
    import baseband_b200 as bb
    from baseband_b200.base.memory import HostBuffer
    nset = int(args.host_gib * 2**30) // (16 * 8032)
    src = HostBuffer(synthetic.vdif_stream(nset, 16, 8000, seed=1))
    n = nset * 32000
    readers = {t: bb.vdif.open(src, 'rs', sample_rate=64e6, dtype=t)
               for t in (torch.float32, torch.float16)}
    outs = {t: torch.empty((n, 16), dtype=t, pin_memory=True)
            for t in readers}
    times = {t: [] for t in readers}
    for t, fh in readers.items():                  # warm-up
        fh.seek(0)
        fh.read(out=outs[t])
    while min(sum(v) for v in times.values()) < args.seconds:
        for t, fh in readers.items():
            fh.seek(0)
            t0 = time.perf_counter()
            fh.read(out=outs[t])
            times[t].append(time.perf_counter() - t0)
    row = {'nsamples': n * 16, 'packed_bytes': nset * 16 * 8032}
    for t, ts in times.items():
        med = float(np.median(ts))
        row[NAMES[t]] = {'gsamples_s_median': n * 16 / med / 1e9,
                         'gsamples_s_best': n * 16 / min(ts) / 1e9,
                         'reads': len(ts)}
    row['float16']['ratio_to_float32_median'] = (
        row['float16']['gsamples_s_median']
        / row['float32']['gsamples_s_median'])
    row['float16']['exact'] = bool(exact(outs[torch.float16],
                                         outs[torch.float32]))
    print(json.dumps({'host_read_C2': row}), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--gib', type=float, default=1.0,
                    help='packed GiB per shape (device-resident decode)')
    ap.add_argument('--host-gib', type=float, default=0.25,
                    help='packed GiB of the host-output read')
    ap.add_argument('--seconds', type=float, default=2.0,
                    help='timed seconds per leg')
    ap.add_argument('--dump', default=None,
                    help='directory for the .npy output dumps')
    ap.add_argument('--out', default=None, help='write the JSON here')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_reduced.py needs a CUDA device')
    if args.dump:
        os.makedirs(args.dump, exist_ok=True)
    dev = torch.device('cuda', torch.cuda.current_device())
    result = {'card': card(), 'device_decode': bench_device(args, dev),
              'host_read': bench_host(args)}
    result['card_after'] = card()
    text = json.dumps(result, indent=1)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text)
    print(text)


if __name__ == '__main__':
    main()
