"""Rate of bb_byte_counts (8-bit state counts) on resident data larger than
L2, against the pure-read probe in the same call, plus tasks.state_counts
against tasks.moments end to end on the same C4 GUPPI stream from pinned
host memory.

    python tools/bench_byte_counts.py [--gib 2] [--reps 10] [--e2e-frames 128]

Prints the GPU name and power limit, then one line per (shape, data): the
rate in GB/s of packed bytes and as a fraction of bb_probe_read, the two
legs alternating.  Nothing is written to the tree."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import baseband_b200 as bb  # noqa: E402
from baseband_b200 import kernels, synthetic, tasks  # noqa: E402
from baseband_b200.base.memory import HostBuffer  # noqa: E402

# (name, nthread, nelem, payload bytes, header bytes before each unit)
SHAPES = [
    ('mwa_vdif_1thread', 1, 2, 512, 32),
    ('mwa_vdif_16thread', 16, 2, 512, 32),
    ('guppi_c4_chanfirst', 512, 4, 4096 * 2 * 2, 0),
    ('guppi_timefirst_2048', 1, 2048, 4096 * 512 * 2 * 2, 6400),
    ('gsb_phased_1024', 2, 1024, 8192, 0),
    # a DADA chunk piece: the payload is one unit, counted in one call
    ('dada_piece_one_unit', 1, 4, 2**31, 0),
]


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(
            ['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm',
             '--format=csv,noheader', '-i', '0'],
            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = 'unknown'
    return name, out


def make_data(nbytes, dist, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    if dist == 'uniform':
        return torch.randint(0, 256, (nbytes,), dtype=torch.uint8,
                             device=dev, generator=g)
    x = torch.randn(nbytes, device=dev, generator=g) * 2.0
    return x.round().to(torch.int8).view(torch.uint8)


def time_legs(legs, reps):
    """Median time of every leg, the legs alternating rep by rep."""
    times = {k: [] for k in legs}
    for _ in range(reps):
        for k, fn in legs.items():
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) * 1e-3)
    return {k: float(np.median(v)) for k, v in times.items()}


def kernel_legs(args, dev):
    for name, nthread, nelem, payload, hdr in SHAPES:
        frame = payload + hdr
        nset = max(1, int(args.gib * 2**30) // (frame * nthread))
        nbytes = nset * nthread * frame
        uo = (torch.arange(nset * nthread, dtype=torch.int64, device=dev)
              * frame + hdr)
        nbin = 4
        per_bin = -(-nset // nbin)
        counts = torch.zeros((nbin, nthread, nelem, 256), dtype=torch.int64,
                             device=dev)
        for dist in ('uniform', 'narrow'):
            raw = make_data(nbytes, dist, dev, seed=len(name))

            def count():
                kernels.byte_counts(raw, uo, nset, nthread, payload, nelem,
                                    counts, 0, per_bin)

            def probe():
                kernels.probe_read(raw)

            count()
            probe()
            torch.cuda.synchronize()
            t = time_legs({'count': count, 'read': probe}, args.reps)
            packed = nset * nthread * payload
            rate = packed / t['count'] / 1e9
            read = nbytes / t['read'] / 1e9
            print('{:22s} {:8s} {:9.1f} GB/s packed  read probe {:7.1f} GB/s'
                  '  fraction {:.2f}  ({:.2f} GiB, {:.3f} ms)'.format(
                      name, dist, rate, read, rate / read, packed / 2**30,
                      t['count'] * 1e3), flush=True)
            del raw
        del uo, counts
        torch.cuda.empty_cache()


def e2e_leg(args, dev):
    nframe = args.e2e_frames
    raw, _ = synthetic.guppi_stream(nframe, nchan=512, npol=2,
                                    samples_per_frame=4096, overlap=64)
    src = HostBuffer(raw)
    fh = bb.guppi.open(src, 'rs', device=dev)
    spf = fh.samples_per_frame
    # bins of 32 frames (~0.9 s of C4): the count table (256 entries per
    # element, 4 MiB a bin) stays small against the payload, as it would in use
    per_bin = 32 * spf

    def counts():
        fh.seek(0)
        return tasks.state_counts(fh, per_bin)

    def moments():
        fh.seek(0)
        return tasks.moments(fh, per_bin)

    c = counts()
    n, total, sq = moments()
    lv = tasks.state_levels(fh).astype(np.int64)
    ok = (np.array_equal(c.sum(-1), n)
          and np.array_equal((c * lv).sum(-1), total)
          and np.array_equal((c * lv * lv).sum(-1), sq))
    times = {'state_counts': [], 'moments': []}
    for _ in range(args.e2e_reps):
        for k, fn in (('state_counts', counts), ('moments', moments)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    fh.close()
    packed = nframe * spf * 512 * 2 * 2
    tc = float(np.median(times['state_counts']))
    tm = float(np.median(times['moments']))
    print('e2e C4 GUPPI from pinned host ({:.2f} GiB packed, {} frames): '
          'state_counts {:.1f} GB/s, moments {:.1f} GB/s, ratio {:.3f}; '
          'counts == moments exactly: {}'.format(
              packed / 2**30, nframe, packed / tc / 1e9, packed / tm / 1e9,
              tm / tc, ok), flush=True)
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gib', type=float, default=2.0,
                    help='resident bytes per shape (well above the L2)')
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--e2e-frames', type=int, default=128)
    ap.add_argument('--e2e-reps', type=int, default=7)
    ap.add_argument('--skip-e2e', action='store_true')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device: there is nothing to measure '
                         'on the CPU')
    dev = torch.device('cuda:0')
    name, power = gpu_info()
    print('GPU: {}; power limit, max SM clock: {}'.format(name, power),
          flush=True)
    kernel_legs(args, dev)
    if not args.skip_e2e and not e2e_leg(args, dev):
        raise SystemExit('state_counts and moments disagree')


if __name__ == '__main__':
    main()
