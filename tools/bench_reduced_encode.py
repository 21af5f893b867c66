"""float32 vs float16 / bfloat16 encoder input on the GPU.

    python tools/bench_reduced_encode.py [--gib 1] [--seconds 2]

Device-resident encode of the named shapes (those of tools/bench_reduced.py),
the unit tables built once so that only the encode kernel is timed:
  C1  VDIF, 8 threads, 2 bit, 5000-byte payloads
  C2  VDIF, 16 threads, 2 bit, 8000-byte payloads (the headline shape)
  C3  Mark 4, 64 tracks, fan-out 4, 8 channels (FAST encode)
  C4  GUPPI, 512 channels, 2 pol, 8-bit complex, channels first
  C5  Mark 5B, 16 channels, 2 bit, 1 % invalid frames
Each shape writes --gib of packed output (well beyond the 126 MB L2); its
input is the decode of random packed data, in float32 and rounded to each
16-bit type.  Legs are warmed up and timed with CUDA events in blocks of
about a quarter second, float32 / float16 / bfloat16 blocks alternating,
until every leg has --seconds.  bb_probe_copy is timed in the same run.
Then two public-API legs on C2, float32 against float16, alternating:
``writer.write`` of a pinned host tensor into a HostBuffer sink, and the
round trip ``read(dtype=..., out=pinned, on_device=writer.write)``.

Reports Gsamples/s, the algorithmic TB/s (input bytes read + packed bytes
written), the ratio to float32, and whether every 16-bit output equals the
float32 encode of the widened input; the card's name and power limit are
read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(
    __file__))))
from baseband_b200 import kernels, levels, synthetic  # noqa: E402
from tools.bench_reduced import NAMES, TYPES, card, time_legs  # noqa: E402


def shapes(nbytes, dev):
    """name -> (packed bytes, float32 input, encode(data, dst))."""
    out = {}
    for name, nthread, payload in (('C1_vdif_8thread_2bit', 8, 5000),
                                   ('C2_vdif_16thread_2bit', 16, 8000)):
        frame = payload + 32
        nset = nbytes // (nthread * frame)
        raw = synthetic.vdif_stream_device(nset, nthread, payload, dev,
                                           seed=synthetic.VDIF_SEED)
        uo = (torch.arange(nset * nthread, dtype=torch.int64, device=dev)
              * frame + 32)
        x = kernels.decode_bitfield(raw, uo, nset, nthread, payload, 2, 1,
                                    False, kernels.CODEC_LEVELS,
                                    levels.offset_binary(2))

        def enc(d, dst, uo=uo, nset=nset, nthread=nthread, payload=payload):
            kernels.encode_bitfield(d, dst, uo, nset, nthread, payload, 2, 1,
                                    kernels.QUANT_OFFSET_BINARY)
        out[name] = (raw.numel(), x, enc)
        del raw
    nframe = nbytes // 160000
    raw4 = synthetic.mark4_stream_device(nframe, dev,
                                         seed=synthetic.MARK4_SEED)
    _, uo4 = kernels.mark4_scan(raw4, nframe, 64)
    x4 = kernels.mark4_decode(raw4, uo4, nframe, 8, 4, False,
                              levels.sign_magnitude())

    def c3(d, dst):
        kernels.mark4_encode(d, dst, uo4, nframe, 8, 4, False)
    out['C3_mark4_64track_fanout4'] = (raw4.numel(), x4, c3)
    del raw4
    nchan, npol, spf = 512, 2, 65536
    fbytes = nchan * spf * npol * 2
    nfr = max(1, nbytes // fbytes)
    g = torch.Generator(device=dev).manual_seed(synthetic.GUPPI_SEED)
    rawg = torch.randint(0, 256, (nfr * fbytes,), dtype=torch.uint8,
                         device=dev, generator=g)
    off = torch.arange(nfr, dtype=torch.int64, device=dev) * fbytes
    cb = torch.zeros(nfr, dtype=torch.int64, device=dev)
    ce = torch.full((nfr,), spf * npol, dtype=torch.int64, device=dev)
    oc0 = torch.arange(nfr, dtype=torch.int64, device=dev) * spf * npol
    xg = torch.empty(nfr * fbytes, dtype=torch.float32, device=dev)
    kernels.decode_int8_transposed(rawg, off, nfr, nchan, spf * npol, 2, cb,
                                   ce, oc0, xg)

    def c4(d, dst):
        kernels.encode_int8_transposed(d, dst, off, nfr, nchan, spf * npol,
                                       2)
    out['C4_guppi_512chan_2pol_int8_complex'] = (rawg.numel(), xg, c4)
    del rawg
    nframe5 = nbytes // 10016
    raw5, _ = synthetic.mark5b_stream_device(nframe5, dev,
                                             seed=synthetic.MARK5B_SEED)
    _, uo5 = kernels.mark5b_scan(raw5, nframe5)
    x5 = kernels.decode_bitfield(raw5, uo5, nframe5, 1, 10000, 2, 16, False,
                                 kernels.CODEC_LEVELS, levels.mark5b(2), 0.0)

    def c5(d, dst):
        kernels.encode_bitfield(d, dst, uo5, nframe5, 1, 10000, 2, 16,
                                kernels.QUANT_MARK5B)
    out['C5_mark5b_2bit_16chan_1pct_invalid'] = (raw5.numel(), x5, c5)
    return out


def bench_device(args, dev):
    result = {}
    nbytes = int(args.gib * 2**30)
    for name, (packed, x32, enc) in shapes(nbytes, dev).items():
        n = x32.numel()
        xs = {torch.float32: x32.reshape(-1)}
        for t in TYPES[1:]:
            xs[t] = xs[torch.float32].to(t)
        dsts = {t: torch.zeros(packed, dtype=torch.uint8, device=dev)
                for t in TYPES}
        per_call, total = time_legs(
            {t: (lambda t=t: enc(xs[t], dsts[t])) for t in TYPES},
            args.seconds)
        torch.cuda.synchronize()
        row = {'packed_bytes': packed, 'nsamples': n}
        for t in TYPES:
            s = per_call[t]
            row[NAMES[t]] = {
                'ms_per_call': s * 1e3, 'seconds_timed': total[t],
                'gsamples_s': n / s / 1e9,
                'algo_tb_s': (n * xs[t].element_size() + packed) / s / 1e12,
                'ratio_to_float32': per_call[torch.float32] / s}
            if t != torch.float32:
                # float32 encode of the widened input (exact on the device:
                # the decoded levels are finite)
                want = torch.zeros_like(dsts[t])
                enc(xs[t].float(), want)
                row[NAMES[t]]['exact'] = bool(torch.equal(dsts[t], want))
                del want
        result[name] = row
        print(json.dumps({name: row}), flush=True)
        del xs, dsts, x32
        torch.cuda.empty_cache()
    half = 2**30
    a = torch.empty(half // 4, dtype=torch.float32, device=dev)
    b = torch.zeros_like(a)
    per, _ = time_legs({'copy': lambda: kernels.probe_copy(a, b)},
                       min(args.seconds, 1.0))
    result['bb_probe_copy'] = {'tb_s': 2 * half / per['copy'] / 1e12,
                               'bytes_per_call': 2 * half}
    print(json.dumps({'bb_probe_copy': result['bb_probe_copy']}), flush=True)
    return result


def _alternate(legs, seconds):
    """legs: {key: callable returning elapsed seconds}; alternate until
    every key has ``seconds``; median and best per key."""
    for fn in legs.values():                       # warm-up
        fn()
    times = {k: [] for k in legs}
    while min(sum(v) for v in times.values()) < seconds:
        for k, fn in legs.items():
            times[k].append(fn())
    return times


def bench_host(args, dev):
    """C2 through the public API: write of a pinned host tensor, and the
    read -> on_device -> write round trip, float32 against float16."""
    import baseband_b200 as bb
    from baseband_b200.base.memory import HostBuffer
    nset = int(args.host_gib * 2**30) // (16 * 8032)
    raw = synthetic.vdif_stream(nset, 16, 8000, seed=1)
    src = HostBuffer(raw)
    n = nset * 32000
    with bb.vdif.open(src, 'rs', sample_rate=64e6) as fh:
        header0 = fh.header0
        x32 = torch.from_numpy(fh.read()).pin_memory()
    host = {torch.float32: x32, torch.float16: x32.to(torch.float16)
            .pin_memory()}
    sinks = {}

    def write_leg(t):
        sink = HostBuffer(raw.size)
        fw = bb.vdif.open(sink, 'ws', header0=header0, nthread=16,
                          sample_rate=64e6, device=dev)
        t0 = time.perf_counter()
        fw.write(host[t])
        fw.close()
        el = time.perf_counter() - t0
        sinks[t] = sink
        return el

    readers = {t: bb.vdif.open(src, 'rs', sample_rate=64e6, dtype=t,
                               device=dev) for t in host}
    outs = {t: torch.empty((n, 16), dtype=t, pin_memory=True) for t in host}
    rsinks = {}

    def round_trip_leg(t):
        fh = readers[t]
        fh.seek(0)
        sink = HostBuffer(raw.size)
        fw = bb.vdif.open(sink, 'ws', header0=header0, nthread=16,
                          sample_rate=64e6, device=dev)
        t0 = time.perf_counter()
        fh.read(out=outs[t], on_device=fw.write)
        fw.close()
        el = time.perf_counter() - t0
        rsinks[t] = sink
        return el

    result = {}
    for leg, fn, sk in (('host_write_C2', write_leg, sinks),
                        ('round_trip_C2', round_trip_leg, rsinks)):
        times = _alternate({t: (lambda t=t, fn=fn: fn(t)) for t in host},
                           args.seconds)
        row = {'nsamples': n * 16, 'packed_bytes': int(raw.size)}
        for t, ts in times.items():
            med = float(np.median(ts))
            row[NAMES[t]] = {'gsamples_s_median': n * 16 / med / 1e9,
                             'gsamples_s_best': n * 16 / min(ts) / 1e9,
                             'calls': len(ts)}
        row['float16']['ratio_to_float32_median'] = (
            row['float16']['gsamples_s_median']
            / row['float32']['gsamples_s_median'])
        row['float16']['same_bytes'] = bool(np.array_equal(
            np.asarray(sk[torch.float16].getvalue()),
            np.asarray(sk[torch.float32].getvalue())))
        result[leg] = row
        print(json.dumps({leg: row}), flush=True)
    return result


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--gib', type=float, default=1.0,
                    help='packed output GiB per shape (device encode)')
    ap.add_argument('--host-gib', type=float, default=0.25,
                    help='packed GiB of the public-API legs')
    ap.add_argument('--seconds', type=float, default=2.0,
                    help='timed seconds per leg')
    ap.add_argument('--out', default=None, help='write the JSON here')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_reduced_encode.py needs a CUDA device')
    dev = torch.device('cuda', torch.cuda.current_device())
    result = {'card': card(), 'device_encode': bench_device(args, dev),
              'public_api': bench_host(args, dev)}
    result['card_after'] = card()
    text = json.dumps(result, indent=1)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text)
    print(text)


if __name__ == '__main__':
    main()
