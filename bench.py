#!/usr/bin/env python
"""Benchmark of the baseband hot path on B200 (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--dump-outputs DIR]

Workload = BASELINE.json configs[1]: synthetic VDIF, 2-bit real, 16 threads,
8032-byte frames; one step = the hot path over `--passes` (default 32)
resident chunks of the 64 GiB logical stream, i.e. 32 GiB of packed frames
per GPU and step: header scan (validity + thread slots + frame-index check)
-> decode to float32 (nsample, 16) -> encode_2bit round trip back to packed
payloads, chunk after chunk.  A chunk (default 1 GiB packed -> 16 GiB
decoded, far larger than the 126 MB L2) is resident in HBM when the timed
region starts.  The default 20 steps keep the GPU busy for ~3.5 s, so the
headline is a SUSTAINED rate (clocks settled under the power cap), not a
burst; the burst figure (best single launch) is printed next to it.  With N
GPUs each rank takes its own contiguous range of frame sets (weak scaling, no
collective on the data path); value = total decoded samples / max-over-ranks
time.

Printed JSON line: see the task contract.  Extra keys: `roofline` (decode
kernel, CUDA-event timed inside the timed region), `cpu_baseline` (numpy
oracle = port of the reference's CPU path, bounded sample, rank 0 at N=1),
`e2e` (public API, pinned host buffers on both ends: `read(out=host array,
on_device=writer.write)` = chunked H2D -> scan+decode -> D2H of the decoded
samples, with every decoded chunk re-encoded in HBM and its frames copied
back),
`clocks`, `gpu_launches`, `sharded_read` (parallel.read_sharded of ONE logical
pinned-host stream over the N ranks, device output, and the optional NCCL
gather in GB/s per GPU) and `consumer` (a second end-to-end line: packed
frames -> state counts / power on the GPU, nothing but the counts returned).

`--impl reference` times the reference's own CPU algorithm (the numpy oracle,
a function-by-function port: astropy is not installable here so the package
itself cannot be imported on the box) on all host cores, same metric/config.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NTHREAD = 16
PAYLOAD = 8000
FRAME = PAYLOAD + 32
SPF = PAYLOAD * 4                    # samples per thread-frame (2 bit)
SET_BYTES = NTHREAD * FRAME          # 128 512
SET_SAMPLES = SPF * NTHREAD          # 512 000 decoded floats
ALGO_BYTES_PER_SAMPLE = (SET_BYTES + SET_SAMPLES * 4) / SET_SAMPLES  # 4.251
LOGICAL_STREAM_BYTES = 64 << 30
_REAL_STDOUT = sys.stdout
METRIC = 'decoded Gsamples/s (device-resident)'
UNIT = 'Gsamples/s'


def config_dict(chunk_bytes, ngpu, passes=1):
    return {
        'workload': 'synthetic VDIF 2-bit real, 16 threads, 8032-byte frames '
                    '(BASELINE.json configs[1]): header scan + decode + '
                    'encode_2bit round trip; a step = {} resident chunks '
                    'per GPU'.format(passes),
        'logical_stream_bytes': LOGICAL_STREAM_BYTES,
        'chunks_per_step': int(passes),
        'packed_bytes_per_gpu_per_step': int(chunk_bytes) * int(passes),
        'chunk_bytes_per_gpu': int(chunk_bytes),
        'frame_sets_per_chunk': int(chunk_bytes // SET_BYTES),
        'decoded_bytes_per_chunk': int(chunk_bytes // SET_BYTES
                                       * SET_SAMPLES * 4),
        'parallelism': 'frame-set ranges x{} (no collective)'.format(ngpu),
        'cache': 'inputs+outputs per step (>= 17 GiB) far exceed the 126 MB '
                 'L2; no flush needed',
    }


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)['hbm_gbs']), 'measured'
    return 6650.0, 'fallback'


# --------------------------------------------------------------- CPU legs
def _cpu_round_trip(nset, seed):
    """Reference CPU path on ``nset`` frame sets: struct-free header parse,
    LUT decode with thread interleave, encode_2bit round trip."""
    from baseband_b200 import synthetic
    from oracle import codec, stream
    raw = synthetic.vdif_stream(nset, NTHREAD, PAYLOAD, seed=seed)
    t0 = time.perf_counter()
    data = stream.vdif_read(raw)                       # (nset*SPF, 16, 1)
    back = np.empty((nset, NTHREAD, PAYLOAD), np.uint8)
    for s in range(nset):
        block = data[s * SPF:(s + 1) * SPF, :, 0]
        for t in range(NTHREAD):
            back[s, t] = codec.vdif_encode(
                np.ascontiguousarray(block[:, t]), 2)
    dt = time.perf_counter() - t0
    return data.shape[0] * NTHREAD, dt


def _cpu_worker(args):
    return _cpu_round_trip(*args)


def cpu_baseline(nset=960):
    nsamp, dt = _cpu_round_trip(nset, 1)
    return {'value': nsamp / dt / 1e9, 'unit': UNIT, 'cores': 1,
            'kind': 'port',
            'sample': '{} frame sets ({:.1f} MB packed) of the same '
                      'synthetic stream, decode + encode round trip, numpy '
                      'oracle'.format(nset, nset * SET_BYTES / 1e6)}


def run_reference(args):
    """--impl reference: the CPU algorithm on all host cores."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = min(os.cpu_count() or 1, 64)
    nset = 32
    ctx = mp.get_context('fork')
    with ctx.Pool(cores) as pool:
        for _ in range(args.warmup):
            pool.map(_cpu_worker, [(2, i) for i in range(cores)])
        t0 = time.perf_counter()
        nsamp = 0
        for k in range(args.steps):
            res = pool.map(_cpu_worker, [(nset, 100 * k + i)
                                         for i in range(cores)])
            nsamp += sum(r[0] for r in res)
        dt = time.perf_counter() - t0
    value = nsamp / dt / 1e9
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT,
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        # the same workload description as the B200 arm prints; what one
        # step of THIS arm covers of it is stated in cpu_baseline.sample
        'config': config_dict(
            int(args.chunk_gib * 2**30) // SET_BYTES * SET_BYTES, args.gpus,
            max(1, args.passes)),
        'cpu_baseline': {
            'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
            'sample': 'a step of this arm is a bounded sample of the '
                      'workload: {} processes x {} frame sets ({:.0f} MB '
                      'packed) of the same synthetic stream, decode + encode '
                      'round trip, numpy oracle (port of the reference CPU '
                      'path; the reference package needs astropy, absent '
                      'here)'.format(cores, nset,
                                     cores * nset * SET_BYTES / 1e6)},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)


# --------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled every ~5 ms through NVML in a
    background thread while the timed region runs."""
    BAD = {'hw_slowdown': 0x8, 'hw_thermal_slowdown': 0x40,
           'sw_thermal_slowdown': 0x20, 'sw_power_cap': 0x4}

    def __init__(self, index):
        self.index = index
        self.sm, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self.thread = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES when mapping the torch index
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            index = self.index
            if visible:
                ids = [v for v in visible.split(',') if v.strip() != '']
                if index < len(ids) and ids[index].strip().isdigit():
                    index = int(ids[index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml = pynvml
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(
                self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nvml
        while not self._stop.is_set():
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.handle,
                                                         nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                for name, bit in self.BAD.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        if self.thread is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [],
                    'samples': 0}
        self._stop.set()
        self.thread.join(timeout=2)
        sm = sorted(self.sm)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None,
                'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(sm)}


# --------------------------------------------------------------- GPU arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    from baseband_b200 import kernels, levels, synthetic

    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if world != args.gpus and world > 1:
        raise SystemExit('--gpus must equal WORLD_SIZE under torchrun')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    from baseband_b200 import device as bb_device
    numa_cpus = bb_device.bind_host_to_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    chunk_bytes = int(args.chunk_gib * 2**30)
    nset = chunk_bytes // SET_BYTES
    nframe = nset * NTHREAD
    chunk_bytes = nset * SET_BYTES
    first_set = rank * (LOGICAL_STREAM_BYTES // SET_BYTES // max(world, 1))
    raw = synthetic.vdif_stream_device(nset, NTHREAD, PAYLOAD, dev,
                                       seed=synthetic.VDIF_SEED + rank,
                                       first_set=first_set)
    slot = torch.full((1024,), -1, dtype=torch.int32, device=dev)
    slot[:NTHREAD] = torch.arange(NTHREAD, dtype=torch.int32, device=dev)
    lv = levels.offset_binary(2)
    out = torch.empty((nset * SPF, NTHREAD, 1), dtype=torch.float32,
                      device=dev)
    back = torch.empty_like(raw)
    back.view(nframe, FRAME)[:, :32] = raw.view(nframe, FRAME)[:, :32]
    dec_events = []
    passes = max(1, args.passes)
    # frame-index check of the scan: the synthetic headers count 2000 frame
    # sets per second from second 100 (synthetic.vdif_headers)
    check = (first_set, 100, 0, 2000)

    def one_pass(record=False):
        _, uo, bad = kernels.vdif_scan(raw, nframe, FRAME, 32, NTHREAD, slot,
                                       NTHREAD, check=check, bad=counter,
                                       want_fields=False)
        if record:
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
        kernels.decode_bitfield(raw, uo, nset, NTHREAD, PAYLOAD, 2, 1, False,
                                kernels.CODEC_LEVELS, lv, out=out)
        if record:
            e1.record()
            dec_events.append((e0, e1))
        kernels.encode_bitfield(out, back, uo, nset, NTHREAD, PAYLOAD, 2, 1,
                                kernels.QUANT_OFFSET_BINARY)
        return uo

    def step(record=False):
        # record one decode launch in four: 640 event pairs would do no harm,
        # but the sustained figure needs no more
        for k in range(passes):
            uo = one_pass(record and (k % 4 == 0))
        return uo

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    counter = kernels.new_counter(dev)
    one_pass()
    torch.cuda.synchronize()
    assert int(counter.item()) == 0
    if not torch.equal(back, raw):
        raise SystemExit('round trip mismatch: decode->encode must be exact')
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = kernels.launch_count
    barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        uo = step(record=True)
    t1.record()
    barrier()
    elapsed_ms = t0.elapsed_time(t1)
    launches = kernels.launch_count - launches0
    clocks = sampler.stop() if rank == 0 else None
    assert int(counter.item()) == 0
    # before measure_ceilings, which overwrites `out`
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, back, uo, nset)
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    dec_all = [a.elapsed_time(b) for a, b in dec_events]
    dec_ms = sum(dec_all) / len(dec_all)          # sustained: mean over the run
    dec_best_ms = min(dec_all)                    # burst: best single launch

    # ------------------------------------------------ ceilings, same run
    ceilings = measure_ceilings(dev, out, kernels)

    # ------------------------------------------------ end-to-end (host bufs)
    e2e = measure_e2e(args, dev, rank, world, lv, slot)
    del out, back, raw
    torch.cuda.empty_cache()
    # the legs beside the contract's numbers must not cost the line itself
    named = _leg(measure_named_configs, args, dev, rank, world)
    sharded = _leg(measure_sharded_read, args, dev, rank, world)
    consumer = _leg(measure_consumer, args, dev, rank, world)
    file_ingest = _leg(measure_file_ingest, args, dev, rank, world)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    samples_per_step = nset * SET_SAMPLES * world * passes
    value = samples_per_step * args.steps / (elapsed_ms * 1e-3) / 1e9
    peak, which = peaks()
    algo_bytes = nset * (SET_BYTES + SET_SAMPLES * 4)
    achieved = algo_bytes / (dec_ms * 1e-3) / 1e9
    burst = algo_bytes / (dec_best_ms * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic(DECODE_KERNEL, nset * SET_SAMPLES)
    wp = ceilings['write_peak_sustained_gbs']
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world,
        'steps': args.steps, 'warmup': max(args.warmup, 3),
        'ms_per_step': elapsed_ms / args.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': config_dict(chunk_bytes, world, passes),
        'timed_region_s': elapsed_ms * 1e-3,
        'decode_only_gsamples_s': nset * SET_SAMPLES / (dec_ms * 1e-3) / 1e9,
        'roofline': {
            'bound': 'hbm', 'kernel': DECODE_KERNEL,
            'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
            'frac': achieved / peak, 'peak_source': which + ' copy bandwidth '
            '(MEASURED_PEAKS.json)',
            'what': 'sustained: mean of {} decode launches spread over the '
                    '{:.1f} s timed region'.format(len(dec_all),
                                                   elapsed_ms * 1e-3),
            'burst': {'achieved': burst, 'frac': burst / peak,
                      'what': 'best single decode launch of the same run'},
            'write_peak': wp, 'frac_of_write_peak': achieved / wp,
            'frac_of_expand_ceiling': achieved
            / ceilings['expand_1to16_sustained_gbs'],
            'ceilings_in_run': ceilings,
            'algorithmic_bytes_per_sample': ALGO_BYTES_PER_SAMPLE,
            'algorithmic_bytes_per_launch': algo_bytes,
            'traffic': traffic, 'traffic_source': traffic_src},
        'e2e': e2e, 'gpu_launches': launches, 'clocks': clocks,
        'named_configs': named, 'sharded_read': sharded,
        'consumer': consumer, 'file_ingest': file_ingest,
        'host_binding': ('rank pinned to the {} CPUs local to its GPU'
                         .format(len(numa_cpus)) if numa_cpus else 'none'),
    }
    if world == 1 and not args.no_cpu_baseline:
        line['cpu_baseline'] = cpu_baseline()
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


DECODE_KERNEL = 'k_decode_bitfield<2,LEVELS,ROWGROUP4>'
DUMP_SETS = 16          # frame sets sampled by --dump-outputs (~42 MB in all)


def dump_outputs(folder, out, back, uo, nset):
    """What the last timed pass hands its caller, as float32 / float64 .npy
    files, so that two builds can be compared output for output: the unit
    offsets of the header scan in full, and the decoded samples and
    re-encoded frames of DUMP_SETS frame sets drawn with a fixed seed (a
    chunk decodes to 16 GiB).  The inputs come from fixed seeds too."""
    import torch
    os.makedirs(folder, exist_ok=True)
    sets = np.sort(np.random.default_rng(0).choice(
        nset, min(DUMP_SETS, nset), replace=False))
    rows = torch.from_numpy(sets).to(out.device)
    arrays = {
        'frame_sets': sets.astype(np.float64),
        'unit_offsets': uo.cpu().numpy().astype(np.float64),
        'decoded': out.view(nset, SPF, NTHREAD)[rows].cpu().numpy(),
        'encoded_frames': back.view(nset, SET_BYTES)[rows].cpu().numpy()
        .astype(np.float32),
    }
    for name, array in arrays.items():
        np.save(os.path.join(folder, name + '.npy'), array)


def _leg(fn, *a):
    """Run one of the additional measurements; a failure is reported in its
    place (and on stderr) instead of ending the run."""
    try:
        return fn(*a)
    except Exception as exc:            # noqa: BLE001 - reported, not hidden
        import traceback
        traceback.print_exc()
        return {'error': '{}: {}'.format(type(exc).__name__, exc)}


def measure_ceilings(dev, scratch, kernels, seconds=0.4):
    """Pure-write and copy rates of this GPU, measured in this run with the
    library's own probe kernels (full-grid st.global.v4 fill; ld/st.v4 copy)
    on the decode output buffer: the ceilings the decode rate is quoted
    against next to MEASURED_PEAKS.json's torch copy figure."""
    import torch
    flat = scratch.view(-1)
    half = flat.numel() // 2
    a, b = flat[:half], flat[half:2 * half]

    def rate(fn, nbytes):
        fn()
        torch.cuda.synchronize(dev)
        ev, t_end = [], time.perf_counter() + seconds
        while time.perf_counter() < t_end:
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            ev.append((e0, e1))
            e1.synchronize()
        ms = [x.elapsed_time(y) for x, y in ev]
        return (nbytes / (sum(ms) / len(ms) * 1e-3) / 1e9,
                nbytes / (min(ms) * 1e-3) / 1e9)

    fill_s, fill_b = rate(lambda: kernels.probe_fill(flat, 1),
                          flat.numel() * 4)
    copy_s, copy_b = rate(lambda: kernels.probe_copy(a, b), 2 * half * 4)
    # 1:16 expansion with ideal access patterns: the first 15/16 of the
    # buffer written from the last 1/16 read (16 interleaved input streams,
    # the shape of this workload)
    n16 = flat.numel() * 4 // 17 // 4096 * 4096
    src = flat[flat.numel() - n16 // 64:]
    dst = flat[:n16 // 4]
    exp_s, exp_b = rate(lambda: kernels.probe_expand(dst, src, 1),
                        n16 + n16 // 16)
    return {'write_peak_sustained_gbs': fill_s, 'write_peak_burst_gbs': fill_b,
            'copy_sustained_gbs': copy_s, 'copy_burst_gbs': copy_b,
            'expand_1to16_sustained_gbs': exp_s,
            'expand_1to16_burst_gbs': exp_b,
            'how': 'bb_probe_fill (decode store pattern) over the {:.0f} GiB '
                   'decode output buffer, bb_probe_copy half -> half, '
                   'bb_probe_expand (reads 1 byte per 16 written from 16 '
                   'interleaved streams, no arithmetic: the ceiling of a '
                   '2 bit -> float32 stream); mean and best launch over {} s '
                   'each'.format(flat.numel() * 4 / 2**30, seconds)}


# the sources the bit-field decode kernel is compiled from
DECODE_SOURCES = ('bb_bitfield.cu', 'bb_bitfield.cuh', 'bb_bitfield_plan.h',
                  'bb_common.cuh', 'bb_quant.cuh', 'bb_runtime.cuh')


def _source_hash(names=DECODE_SOURCES):
    """Hash of a kernel's sources: ncu figures are only quoted for the code
    they were captured from."""
    import hashlib
    h = hashlib.sha256()
    for name in sorted(names):
        with open(os.path.join(ROOT, 'baseband_b200', 'csrc', name),
                  'rb') as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def ncu_traffic(kernel, nsample):
    """dram bytes per launch of ``kernel`` from the committed ncu capture
    (profiles/ncu_traffic.json, written by tools/ncu_traffic.py from an
    `ncu --set full` report), scaled to this launch's sample count -- or
    None when no capture exists for the kernel sources as they are now."""
    path = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    try:
        with open(path) as fh:
            table = json.load(fh)
        entry = table[kernel]
    except (OSError, KeyError, ValueError):
        return None, 'no ncu capture committed for this kernel'
    if entry.get('csrc_sha16') != _source_hash(
            entry.get('sources', DECODE_SOURCES)):
        return None, ('stale: {} was captured from other kernel sources ({})'
                      .format(entry.get('report'), entry.get('csrc_sha16')))
    per_sample = (entry['dram_bytes_read'] + entry['dram_bytes_write']) \
        / entry['samples_per_launch']
    return per_sample * nsample, '{} ({} B/sample measured x {} samples)' \
        .format(entry.get('report'), round(per_sample, 4), nsample)


def measure_e2e(args, dev, rank, world, lv, slot):
    """End to end through the public API with HOST buffers: pinned host
    frames -> ``vdif.open(..., 'rs', device=dev).read()`` (H2D of the packed
    frames, header scan, decode) -> D2H of the decoded samples (what a numpy
    user of ``read()`` receives) -> ``vdif.open(..., 'ws').write(data)``
    (encode_2bit round trip, D2H of the re-packed frames into a pinned
    host sink).  Every byte crosses PCIe inside the timed region."""
    import torch
    import torch.distributed as dist
    import baseband_b200 as bb
    from baseband_b200 import synthetic
    from baseband_b200.base.memory import HostBuffer
    nset = int(args.e2e_mib * 2**20) // SET_BYTES
    src = HostBuffer(synthetic.vdif_stream(
        nset, NTHREAD, PAYLOAD, seed=7 + rank,
        thread_order=np.arange(NTHREAD)))
    sink = HostBuffer(src.size)
    host_out = torch.empty((nset * SPF, NTHREAD), dtype=torch.float32,
                           pin_memory=True)
    chunk = int(args.e2e_chunk_mib * 2**20)
    reader = bb.vdif.open(src, 'rs', sample_rate=64e6, chunk_nbytes=chunk)
    dev_reader = bb.vdif.open(src, 'rs', sample_rate=64e6, device=dev,
                              chunk_nbytes=chunk)
    host_view = host_out.numpy()

    def step():
        # read() streams the frames through the GPU in chunks (H2D, scan,
        # decode, D2H overlapped); each decoded chunk is also handed to the
        # writer while it is still in HBM (encode + D2H of the frames).
        reader.seek(0)
        sink.seek(0)
        writer = bb.vdif.open(sink, 'ws', header0=reader.header0,
                              nthread=NTHREAD, sample_rate=64e6, device=dev)
        reader.read(out=host_view, on_device=writer.write)
        writer._flush(final=False)
        torch.cuda.synchronize(dev)

    for _ in range(2):
        step()
    if world > 1:
        dist.barrier()
    steps = max(2, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    ok = bool(np.array_equal(sink.getvalue(), src.getvalue()))

    # Device-output option: same ingest, decoded samples stay in HBM for a
    # consumer on the GPU; only a spot value is read back.
    def step_dev():
        dev_reader.seek(0)
        data = dev_reader.read()
        return float(data[-1, -1].item())

    step_dev()
    t1 = time.perf_counter()
    for _ in range(steps):
        step_dev()
    dt_dev = time.perf_counter() - t1

    # Link rates for context: plain pinned <-> device copies of the same
    # buffers (what PCIe delivers on this box).
    def copy_rate(dst, srcbuf):
        # all ranks copy at the same time (barrier first), slowest rank's rate:
        # the link as the e2e pipeline finds it, not an idle one
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        dst.copy_(srcbuf, non_blocking=True)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        e0.record()
        for _ in range(3):
            dst.copy_(srcbuf, non_blocking=True)
        e1.record()
        torch.cuda.synchronize(dev)
        rate = 3 * srcbuf.numel() * srcbuf.element_size() / (
            e0.elapsed_time(e1) * 1e-3) / 1e9
        if world > 1:
            t = torch.tensor([rate], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            rate = float(t.item())
        return rate

    probe = torch.empty_like(host_out, device=dev)
    d2h_gbs = copy_rate(host_out, probe)
    h2d_gbs = copy_rate(probe, host_out)
    del probe
    if world > 1:
        t = torch.tensor([dt], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    return {'value': nset * SET_SAMPLES * world * steps / dt / 1e9,
            'unit': UNIT, 'h2d_bytes_per_step': int(src.size),
            'd2h_bytes_per_step': int(host_out.numel() * 4 + src.size),
            'steps': steps, 'round_trip_exact': ok,
            'device_output_gsamples_s': nset * SET_SAMPLES * steps / dt_dev
            / 1e9,
            'pcie': {
                'h2d_copy_gbs': h2d_gbs, 'd2h_copy_gbs': d2h_gbs,
                'e2e_d2h_gbs': (host_out.numel() * 4 + src.size) * steps
                / dt / 1e9,
                'ingest_h2d_gbs': src.size * steps / dt_dev / 1e9,
                'e2e_fraction_of_d2h_link': (host_out.numel() * 4 + src.size)
                * steps / dt / 1e9 / d2h_gbs,
                'note': 'link rates: plain pinned copies of the same buffers '
                        'with all ranks copying at once (barrier, slowest '
                        'rank).  e2e moves 4 B/sample device->host: '
                        'e2e_d2h_gbs vs d2h_copy_gbs is the fraction of the '
                        'link it reaches; ingest_h2d_gbs is the packed-frame '
                        'ingest rate of the device-output path'},
            'api': "vdif.open(HostBuffer,'rs').read(out=pinned numpy, "
                   "on_device=vdif.open(HostBuffer,'ws').write)",
            'note': 'per GPU {} MiB packed per step; PCIe bound: the decoded '
                    'float32 array returned to the host is 16x the packed '
                    'input'.format(args.e2e_mib)}


def measure_sharded_read(args, dev, rank, world):
    """`parallel.read_sharded` on ONE logical stream held in pinned host
    memory: every rank opens the same frames (same seed) and decodes its
    contiguous share of frame sets to a device tensor -- H2D of the packed
    frames inside the timed region, no collective; then the optional
    gather (`gather=True`): each rank decodes into its place in the full
    result and one in-place all_gather_into_tensor over NVLink fills in the
    rest.  Rates: Gsamples/s over all ranks (max-over-ranks time) and the
    collective alone in GB/s received per GPU (CUDA events)."""
    import torch
    import torch.distributed as dist
    import baseband_b200 as bb
    from baseband_b200 import parallel, synthetic
    from baseband_b200.base.memory import HostBuffer
    nbytes = int(args.sharded_mib * 2**20)
    if nbytes <= 0:
        return None
    nset = max(world, nbytes // SET_BYTES)
    src = HostBuffer(synthetic.vdif_stream(
        nset, NTHREAD, PAYLOAD, seed=99, thread_order=np.arange(NTHREAD)))
    fh = bb.vdif.open(src, 'rs', sample_rate=64e6, device=dev,
                      chunk_nbytes=int(args.e2e_chunk_mib * 2**20))
    reps = 3

    def timed(fn):
        fn()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            out = fn()
        torch.cuda.synchronize(dev)
        dt = (time.perf_counter() - t0) / reps
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt, out

    dt, (data, (a, b)) = timed(lambda: parallel.read_sharded(fh, rank, world))
    result = {'logical_stream_bytes': int(src.size),
              'gsamples_s': nset * SET_SAMPLES / dt / 1e9,
              'shard_rows': int(b - a),
              'api': "parallel.read_sharded(vdif.open(HostBuffer, 'rs', "
                     "device=...))"}
    del data
    if world > 1:
        dt, (whole, _) = timed(
            lambda: parallel.read_sharded(fh, rank, world, gather=True))
        result['gather_gsamples_s'] = nset * SET_SAMPLES / dt / 1e9
        # the collective alone, in place on the gathered result
        block = parallel.gather_block(fh, world)
        shape = tuple(whole.shape[1:])
        del whole
        full = torch.empty((world * block,) + shape, dtype=torch.float32,
                           device=dev)
        mine = full[rank * block:(rank + 1) * block]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        dist.all_gather_into_tensor(full, mine)
        torch.cuda.synchronize(dev)
        dist.barrier()
        ev[0].record()
        for _ in range(reps):
            dist.all_gather_into_tensor(full, mine)
        ev[1].record()
        torch.cuda.synchronize(dev)
        ms = ev[0].elapsed_time(ev[1]) / reps
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        recv = (world - 1) * block * NTHREAD * 4
        result['all_gather'] = {
            'ms': float(t.item()),
            'received_gbs_per_gpu': recv / (float(t.item()) * 1e-3) / 1e9,
            'bytes_received_per_gpu': int(recv),
            'how': 'one in-place all_gather_into_tensor of equal frame-'
                   'aligned blocks (NCCL over NVLink), CUDA events, max '
                   'over ranks'}
        del full, mine
    fh.close()
    torch.cuda.empty_cache()
    return result


def measure_file_ingest(args, dev, rank, world):
    """Users open files: the same frames from a FILE in the page cache
    (/dev/shm) through `vdif.open(path, 'rs', device=...).read()`: native
    thread pool copying out of an mmap of the file into pinned staging, H2D,
    scan + decode, samples left in HBM.  Packed GB/s per GPU (slowest rank)
    and Gsamples/s over all ranks."""
    import torch
    import torch.distributed as dist
    import baseband_b200 as bb
    from baseband_b200 import synthetic
    nbytes = int(args.file_mib * 2**20)
    if nbytes <= 0:
        return None
    nset = max(1, nbytes // SET_BYTES)
    folder = '/dev/shm' if os.path.isdir('/dev/shm') else '/tmp'
    path = os.path.join(folder, 'bb_bench_{}_{}.vdif'.format(os.getpid(),
                                                             rank))
    try:
        synthetic.vdif_stream(nset, NTHREAD, PAYLOAD, seed=41 + rank,
                              thread_order=np.arange(NTHREAD)).tofile(path)
        fh = bb.vdif.open(path, 'rs', sample_rate=64e6, device=dev)
        best = None
        for rep in range(9):
            fh.seek(0)
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            data = fh.read()
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            best = dt if best is None or rep and dt < best else best
            del data
        fh.close()
    finally:
        if os.path.exists(path):
            os.remove(path)
    torch.cuda.empty_cache()
    return {'packed_gbs_per_gpu': nset * SET_BYTES / best / 1e9,
            'gsamples_s': nset * SET_SAMPLES * world / best / 1e9,
            'file_bytes': int(nset * SET_BYTES),
            'api': "vdif.open(path, 'rs', device=...).read() of a file in "
                   "the page cache (" + folder + ")",
            'how': 'best of 8 passes after a warm-up, all ranks at once, '
                   'slowest rank; bb_host_copy out of an mmap of the file '
                   '-> pinned staging -> H2D -> scan + decode'}


def measure_consumer(args, dev, rank, world):
    """Second end-to-end line: a consumer that stays on the GPU.  Pinned host
    frames -> `tasks.state_counts(fh, samples_per_bin)` (the reader's ingest
    pipeline: H2D of the packed frames, header scan with frame-index check,
    bb_state_counts on the packed words) -> the counts (a few KB) back on the
    host as a numpy array, from which integrated power follows.  No float32
    sample ever exists, so the rate is set by the H2D link at 2 bits per
    sample instead of the D2H link at 32.  Also the kernel alone on a
    resident chunk, in GB/s of packed bytes read."""
    import torch
    import torch.distributed as dist
    import baseband_b200 as bb
    from baseband_b200 import kernels, synthetic, tasks
    from baseband_b200.base.memory import HostBuffer
    nbytes = int(args.consumer_mib * 2**20)
    if nbytes <= 0:
        return None
    nset = max(1, nbytes // SET_BYTES)
    src = HostBuffer(synthetic.vdif_stream(
        nset, NTHREAD, PAYLOAD, seed=31 + rank,
        thread_order=np.arange(NTHREAD)))
    fh = bb.vdif.open(src, 'rs', sample_rate=64e6, device=dev,
                      chunk_nbytes=int(args.e2e_chunk_mib * 2**20))
    sets_per_bin = 200                     # 0.1 s of this stream per bin

    def step():
        fh.seek(0)
        return tasks.state_counts(fh, sets_per_bin * SPF)

    counts = step()
    assert int(counts.sum()) == nset * SET_SAMPLES
    if world > 1:
        dist.barrier()
    steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(steps):
        counts = step()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    fh.close()
    # the kernel alone, chunk resident in HBM
    kset = int(args.chunk_gib * 2**30) // SET_BYTES
    raw = synthetic.vdif_stream_device(kset, NTHREAD, PAYLOAD, dev,
                                       seed=synthetic.VDIF_SEED + rank)
    uo = (torch.arange(kset * NTHREAD, dtype=torch.int64, device=dev)
          * FRAME + 32)
    acc = torch.zeros((-(-kset // sets_per_bin), NTHREAD, 1, 4),
                      dtype=torch.int64, device=dev)
    ev = []
    for k in range(8):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        kernels.state_counts(raw, uo, kset, NTHREAD, PAYLOAD, 2, 1, acc,
                             sets_per_bin=sets_per_bin)
        e1.record()
        ev.append((e0, e1))
    torch.cuda.synchronize(dev)
    ms = sorted(a.elapsed_time(b) for a, b in ev[2:])
    kms = ms[len(ms) // 2]
    # its ceiling, in the same run: the pure-read probe over the same bytes
    ev = []
    whole = raw[:raw.numel() // 16 * 16]
    for k in range(8):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        kernels.probe_read(whole)
        e1.record()
        ev.append((e0, e1))
    torch.cuda.synchronize(dev)
    ms = sorted(a.elapsed_time(b) for a, b in ev[2:])
    read_peak = whole.numel() / (ms[len(ms) // 2] * 1e-3) / 1e9
    frame_gbs = kset * NTHREAD * FRAME / (kms * 1e-3) / 1e9
    del raw, uo, acc, whole
    torch.cuda.empty_cache()
    return {'value': nset * SET_SAMPLES * world * steps / dt / 1e9,
            'unit': UNIT, 'h2d_bytes_per_step': int(src.size),
            'd2h_bytes_per_step': int(counts.nbytes), 'steps': steps,
            'ingest_h2d_gbs_per_gpu': src.size * steps / dt / 1e9,
            'api': "tasks.state_counts(vdif.open(HostBuffer, 'rs', "
                   "device=...), samples_per_bin) -> numpy int64 "
                   "(nbin, 16, 4); tasks.integrated_power from the same",
            'kernel': {
                'name': 'k_state_counts_reg<2,1>',
                'packed_gbs': kset * NTHREAD * PAYLOAD / (kms * 1e-3) / 1e9,
                'gsamples_s': kset * SET_SAMPLES / (kms * 1e-3) / 1e9,
                'ms': kms, 'bound': 'hbm read',
                'read_peak_gbs': read_peak,
                'frac_of_read_peak': frame_gbs / read_peak,
                'what': 'bb_state_counts alone on a resident {:.1f} GiB '
                        'chunk (median of 6 launches, CUDA events); bytes = '
                        'payload bytes read; read_peak = bb_probe_read over '
                        'the same buffer (a kernel that loads and stores '
                        'nothing), the fraction counts whole frames, as the '
                        'headers share sectors with the payloads'.format(
                            args.chunk_gib)},
            'note': 'packed frames in, state counts out: what '
                    'Integrate(Square(fh)) needs, without the 16x expansion '
                    'to float32 ever touching HBM or PCIe'}


def measure_named_configs(args, dev, rank, world):
    """Device-resident header scan + decode of the other shapes BASELINE.json
    names (configs[2..4]; SURVEY.md 8(d) C3-C5), outside the headline timed
    region: per-GPU chunk resident in HBM, CUDA events around each pass, max
    over ranks, Gsamples/s summed over ranks, GB/s = (frame bytes read +
    float32 written) / time per GPU against the measured copy peak."""
    import torch
    import torch.distributed as dist
    from baseband_b200 import kernels, levels, synthetic
    peak, _ = peaks()
    nbytes = int(args.named_mib * 2**20)
    if nbytes <= 0:
        return None
    steps = max(3, min(args.steps, 10))
    result = {}

    def timed(name, fn, algo_bytes, nsamp, note):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        ev = [(torch.cuda.Event(enable_timing=True),
               torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in ev:
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize(dev)
        ms = sum(a.elapsed_time(b) for a, b in ev) / steps
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        gbs = algo_bytes / (ms * 1e-3) / 1e9
        result[name] = {'gsamples_s': nsamp * world / (ms * 1e-3) / 1e9,
                        'hbm_gbs_per_gpu': gbs, 'frac': gbs / peak,
                        'ms_per_pass': ms, 'chunk_bytes_per_gpu': algo_bytes
                        - 4 * nsamp, 'what': note}

    # C3: Mark 4, 64 tracks, fan-out 4, 2 bit, 8 channels
    nframe = max(1, nbytes // 160000)
    raw = synthetic.mark4_stream_device(nframe, dev,
                                        seed=synthetic.MARK4_SEED + rank)
    out = torch.empty((nframe * 80000, 8), dtype=torch.float32, device=dev)
    lv4 = levels.sign_magnitude()

    def c3():
        _, uo = kernels.mark4_scan(raw, nframe, 64)
        kernels.mark4_decode(raw, uo, nframe, 8, 4, False, lv4, out=out)

    timed('C3_mark4_64track_fanout4', c3, raw.numel() + out.numel() * 4,
          out.numel(), 'bb_mark4_scan + bb_mark4_decode (track reorder, '
          'header-overwritten rows -> fill)')
    del raw, out
    torch.cuda.empty_cache()

    # C4: GUPPI 8-bit complex, 2 pol, 512 channels, channels first, overlap
    nchan, npol, spf, ov = 512, 2, 65536, 512
    fbytes = nchan * spf * npol * 2
    nfr = max(1, nbytes // fbytes)
    g = torch.Generator(device=dev).manual_seed(synthetic.GUPPI_SEED + rank)
    raw = torch.randint(0, 256, (nfr * fbytes,), dtype=torch.uint8,
                        device=dev, generator=g)
    off = torch.arange(nfr, dtype=torch.int64, device=dev) * fbytes
    cb = torch.zeros(nfr, dtype=torch.int64, device=dev)
    ce = torch.full((nfr,), (spf - ov) * npol, dtype=torch.int64, device=dev)
    ce[-1] = spf * npol
    oc0 = torch.cumsum(ce - cb, 0) - (ce - cb)
    ncols = int((ce - cb).sum().item())
    out = torch.empty((ncols * nchan * 2,), dtype=torch.float32, device=dev)
    timed('C4_guppi_512chan_2pol_int8_complex',
          lambda: kernels.decode_int8_transposed(
              raw, off, nfr, nchan, spf * npol, 2, cb, ce, oc0, out),
          out.numel() * 5, out.numel(),
          'bb_decode_int8_transposed (channels-first -> (time, pol, chan) '
          'complex64, overlap columns skipped; bytes count non-overlap input)')
    del raw, out
    torch.cuda.empty_cache()

    # C5: Mark 5B 2 bit, 16 channels, 1 % invalid (fill pattern) frames
    nframe = max(1, nbytes // 10016)
    raw, valid = synthetic.mark5b_stream_device(
        nframe, dev, seed=synthetic.MARK5B_SEED + rank)
    out = torch.empty((nframe * 2500, 16), dtype=torch.float32, device=dev)
    lv5 = levels.mark5b(2)

    def c5():
        fields, uo = kernels.mark5b_scan(raw, nframe)
        kernels.decode_bitfield(raw, uo, nframe, 1, 10000, 2, 16, False,
                                kernels.CODEC_LEVELS, lv5, -999.0, out=out)
        return fields

    timed('C5_mark5b_2bit_16chan_1pct_invalid', c5,
          raw.numel() + out.numel() * 4, out.numel(),
          'bb_mark5b_scan (BCD fields, fill-pattern validity) + '
          'bb_decode_bitfield with fill_value for invalid frames')
    fields = c5()
    torch.cuda.synchronize(dev)
    got_valid = fields[kernels.M5B_VALID].cpu().numpy().astype(bool)
    filled = (out.view(nframe, -1)[:, 0] == -999.0).cpu().numpy()
    result['C5_mark5b_2bit_16chan_1pct_invalid']['validity_exact'] = bool(
        np.array_equal(got_valid, valid) and np.array_equal(~filled, valid))
    return result


def main():
    # NCCL prints a version banner on stdout when NCCL_DEBUG=VERSION; the
    # contract is ONE JSON line on stdout.
    # Libraries (NCCL's version banner) write to fd 1 behind Python's back:
    # point fd 1 at stderr for the whole run and keep the real stdout for the
    # one JSON line.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--chunk-gib', type=float, default=1.0,
                    help='packed bytes of one resident chunk per GPU')
    ap.add_argument('--passes', type=int, default=32,
                    help='chunks per step (32 x 1 GiB: 20 steps keep the GPU '
                         'busy for ~3.5 s, a sustained figure)')
    ap.add_argument('--e2e-mib', type=float, default=256.0,
                    help='packed MiB per GPU and step of the e2e leg')
    ap.add_argument('--e2e-chunk-mib', type=float, default=32.0,
                    help='packed MiB per pipeline stage of the e2e reader')
    ap.add_argument('--named-mib', type=float, default=1024.0,
                    help='packed MiB per GPU for the C3-C5 shapes (0 = skip)')
    ap.add_argument('--sharded-mib', type=float, default=256.0,
                    help='packed MiB of the ONE logical stream read_sharded '
                         'splits over the ranks (0 = skip)')
    ap.add_argument('--file-mib', type=float, default=512.0,
                    help='packed MiB per GPU of the file-ingest leg (0 = '
                         'skip)')
    ap.add_argument('--consumer-mib', type=float, default=512.0,
                    help='packed MiB per GPU and step of the state-count '
                         'consumer leg (0 = skip)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one '
                         'computed to DIR/<name>.npy (rank 0, B200 arm)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to the b200 implementation')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
