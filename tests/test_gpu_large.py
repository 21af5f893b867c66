"""Parity at BASELINE-like sizes through size-independent properties:
decode -> encode round trips are the identity on the packed bytes, chunked
reads equal one-shot reads, invalid frames are exactly fill, and randomly
chosen frames agree with the oracle."""
import io

import numpy as np
import pytest
import torch

import baseband_b200 as bb
from baseband_b200 import kernels, levels, synthetic
from baseband_b200.base.memory import HostBuffer
from oracle import codec, stream as ostream

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def test_c2_vdif_round_trip_256mib():
    nthread, payload, frame = 16, 8000, 8032
    nset = (256 << 20) // (nthread * frame)
    raw = synthetic.vdif_stream_device(nset, nthread, payload, DEV, seed=99)
    nframe = nset * nthread
    slot = torch.arange(1024, dtype=torch.int32, device=DEV)
    slot[nthread:] = -1
    fields, uo, bad = kernels.vdif_scan(raw, nframe, frame, 32, nthread, slot,
                                        nthread)
    assert int(bad.item()) == 0
    out = kernels.decode_bitfield(raw, uo, nset, nthread, payload, 2, 1,
                                  False, kernels.CODEC_LEVELS,
                                  levels.offset_binary(2))
    back = torch.zeros_like(raw)
    back.view(nframe, frame)[:, :32] = raw.view(nframe, frame)[:, :32]
    kernels.encode_bitfield(out, back, uo, nset, nthread, payload, 2, 1,
                            kernels.QUANT_OFFSET_BINARY)
    assert torch.equal(back, raw)
    # only the four levels occur, equally often within 1 %
    vals, counts = torch.unique(out[:1 << 22], return_counts=True)
    assert vals.numel() == 4
    assert float(counts.max() - counts.min()) / float(counts.sum()) < 0.01
    # randomly chosen thread-frames against the oracle
    rng = np.random.default_rng(0)
    host = raw.view(nframe, frame)
    tid = fields[kernels.VDIF_THREAD_ID].cpu().numpy()
    for i in rng.integers(0, nframe, 12):
        words = host[i, 32:].cpu().numpy().view('<u4')
        want = codec.vdif_payload_decode(words, 2, (1,), False)[:, 0]
        s = i // nthread
        got = out[s * 32000:(s + 1) * 32000, tid[i], 0].cpu().numpy()
        assert np.array_equal(got.view('u4'), want.view('u4'))


def test_c5_mark5b_invalid_frames_large():
    nframe = 20000                                   # 200 MB
    raw, valid = synthetic.mark5b_stream(nframe, invalid_fraction=0.01,
                                         seed=5)
    assert 100 < (~valid).sum() < 320
    src = HostBuffer(raw)
    with bb.mark5b.open(src, 'rs', nchan=16, sample_rate=16e6, kday=56000,
                        fill_value=-999., device=DEV,
                        chunk_nbytes=32 << 20) as fh:
        data = fh.read()
    per = data.view(nframe, 2500 * 16)
    is_fill = (per == -999.).all(1).cpu().numpy()
    assert np.array_equal(is_fill, ~valid)
    assert not bool((per[torch.from_numpy(valid).to(DEV)] == -999.).any())
    for i in np.random.default_rng(1).integers(0, nframe, 8):
        want = ostream.mark5b_read(raw[i * 10016:(i + 1) * 10016], 16,
                                   fill_value=-999.)
        assert np.array_equal(data[i * 2500:(i + 1) * 2500].cpu().numpy(),
                              want)
    # header fields parsed on the GPU for the whole stream
    d_raw = torch.from_numpy(raw).to(DEV)
    fields, uo = kernels.mark5b_scan(d_raw, nframe)
    f = fields.cpu().numpy()
    assert np.array_equal(f[kernels.M5B_FRAME_NR],
                          np.arange(nframe) % 6400)
    assert np.array_equal(f[kernels.M5B_SECONDS],
                          3600 + np.arange(nframe) // 6400)
    assert np.array_equal(f[kernels.M5B_VALID].astype(bool), valid)
    assert np.all(f[kernels.M5B_JDAY] == 123)


def test_c3_mark4_round_trip_large():
    nframe = 1200                                    # 192 MB
    raw = torch.from_numpy(synthetic.mark4_stream(nframe, seed=8)).to(DEV)
    off = torch.arange(nframe, dtype=torch.int64, device=DEV) * 160000 + 1280
    out = kernels.mark4_decode(raw, off, nframe, 8, 4, False,
                               levels.sign_magnitude(), fill_value=7.)
    rows = out.view(nframe, 80000, 8)
    assert bool((rows[:, :640] == 7.).all())
    assert not bool((rows[:, 640:] == 7.).any())
    back = raw.clone()
    back.view(nframe, 160000)[:, 1280:] = 0
    kernels.mark4_encode(out, back, off, nframe, 8, 4, False)
    assert torch.equal(back, raw)
    i = 777
    words = raw.view(nframe, 160000)[i].cpu().numpy().view('<u8')
    want = codec.mark4_decode(words[160:], 8, 4, False)
    assert np.array_equal(rows[i, 640:].cpu().numpy(), want)


def test_c4_guppi_overlap_large():
    raw, truth = synthetic.guppi_stream(6, nchan=512, npol=2,
                                        samples_per_frame=8192, overlap=512,
                                        seed=3)              # 100 MB
    cube = truth.astype(np.float32).transpose(1, 2, 0, 3)
    want = (cube[..., 0] + 1j * cube[..., 1]).astype(np.complex64)
    with bb.guppi.open(io.BytesIO(raw.tobytes()), 'rs', device=DEV,
                       chunk_nbytes=40 << 20) as fh:
        assert fh.shape == want.shape
        data = fh.read()
        assert torch.equal(data, torch.from_numpy(want).to(DEV))
        fh.seek(7000)
        part = fh.read(20000)
        assert torch.equal(part, torch.from_numpy(want[7000:27000]).to(DEV))
    with bb.guppi.open(io.BytesIO(raw.tobytes()), 'rs') as fh:
        fh.seek(100)
        assert np.array_equal(fh.read(9000), want[100:9100])


def test_chunked_equals_one_shot_and_pickle():
    import pickle
    raw = synthetic.vdif_stream(40, 8, 5000, seed=1, invalid=[17])
    a = bb.vdif.open(io.BytesIO(raw.tobytes()), 'rs', sample_rate=32e6,
                     fill_value=3.).read()
    fh = bb.vdif.open(io.BytesIO(raw.tobytes()), 'rs', sample_rate=32e6,
                      fill_value=3., chunk_nbytes=3 * 8 * 5032)
    b = fh.read()
    assert np.array_equal(a, b)
    state = fh.__getstate__()
    assert state['_stages'] is None and state['_streams'] is None


# ---------------------------------------------------------------------------
# BASELINE.json's FULL logical sizes, streamed as 1 GiB resident chunks (the
# way bench.py and the stream readers process them), checked per chunk through
# size-independent properties with exact integer arithmetic:
#   * decode -> encode reproduces the packed bytes (round trip identity);
#   * the number of decoded samples at each level equals the number of
#     payload codes mapping to it (histogram of checksums);
#   * int8 data: the sum of the decoded values equals the sum of the bytes.
def _code_counts_2bit(payload_bytes):
    """Occurrences of the 2-bit codes 0..3 in a uint8 CUDA tensor."""
    hist = torch.bincount(payload_bytes.reshape(-1), minlength=256)
    codes = torch.arange(256, device=hist.device)
    return [int(sum((hist * (((codes >> s) & 3) == c)).sum()
                    for s in (0, 2, 4, 6)).item()) for c in range(4)]


def test_c2_full_64gib_stream():
    nthread, payload, frame = 16, 8000, 8032
    nset = (1 << 30) // (nthread * frame)
    nframe = nset * nthread
    slot = torch.arange(1024, dtype=torch.int32, device=DEV)
    slot[nthread:] = -1
    lv = levels.offset_binary(2)
    out = torch.empty((nset * 32000, nthread, 1), dtype=torch.float32,
                      device=DEV)
    nchunk = (64 << 30) // (nset * nthread * frame)
    total = 0
    # the consumer alongside: state counts of the whole stream in bins of
    # 10 000 frame sets that do not line up with the chunks
    per_bin = 10000
    counts = kernels.zeros((-(-nchunk * nset // per_bin), nthread, 1, 4),
                           torch.int64, torch.device(DEV))
    for k in range(nchunk):
        raw = synthetic.vdif_stream_device(nset, nthread, payload, DEV,
                                           seed=1000 + k, first_set=k * nset)
        _, uo, bad = kernels.vdif_scan(raw, nframe, frame, 32, nthread, slot,
                                       nthread)
        kernels.decode_bitfield(raw, uo, nset, nthread, payload, 2, 1, False,
                                kernels.CODEC_LEVELS, lv, out=out)
        back = torch.zeros_like(raw)
        back.view(nframe, frame)[:, :32] = raw.view(nframe, frame)[:, :32]
        kernels.encode_bitfield(out, back, uo, nset, nthread, payload, 2, 1,
                                kernels.QUANT_OFFSET_BINARY)
        assert int(bad.item()) == 0
        assert torch.equal(back, raw), 'chunk %d' % k
        kernels.state_counts(raw, uo, nset, nthread, payload, 2, 1, counts,
                             set_origin=k * nset, sets_per_bin=per_bin)
        if k % 8 == 0:          # histogram check on every 8th chunk
            want = _code_counts_2bit(raw.view(nframe, frame)[:, 32:])
            got = [int((out == float(v)).sum().item()) for v in lv]
            assert got == want, 'chunk %d' % k
            one = kernels.zeros((1, nthread, 1, 4), torch.int64,
                                torch.device(DEV))
            kernels.state_counts(raw, uo, nset, nthread, payload, 2, 1, one)
            assert one.sum((0, 1, 2)).tolist() == want, 'chunk %d' % k
            per_thread = torch.stack([(out[:, :, 0] == float(v)).sum(0)
                                      for v in lv], -1)
            assert torch.equal(one[0, :, 0], per_thread), 'chunk %d' % k
        total += out.numel()
        del raw, back
    assert total >= 2.7e11          # the 64 GiB stream: 2.74e11 samples
    # every sample of the stream was counted exactly once, bin by bin
    assert int(counts.sum().item()) == total
    per = counts.sum((1, 2, 3)).cpu().numpy()
    assert (per[:-1] == per_bin * 32000 * nthread).all()
    assert per[-1] == total - per[:-1].sum()


def test_c3_full_16gib_mark4_stream():
    nframe = (1 << 30) // 160000
    lv = levels.sign_magnitude()
    out = torch.empty((nframe * 80000, 8), dtype=torch.float32, device=DEV)
    for k in range(16):
        raw = synthetic.mark4_stream_device(nframe, DEV, seed=2000 + k)
        _, uo = kernels.mark4_scan(raw, nframe, 64)
        kernels.mark4_decode(raw, uo, nframe, 8, 4, False, lv, fill_value=9.,
                             out=out)
        back = raw.clone()
        back.view(nframe, 160000)[:, 1280:] = 0
        kernels.mark4_encode(out, back, uo, nframe, 8, 4, False)
        assert torch.equal(back, raw), 'chunk %d' % k
        rows = out.view(nframe, 80000, 8)
        assert bool((rows[:, :640] == 9.).all())
        if k % 4 == 0:
            # sign bits even, magnitude bits odd tracks: every payload bit
            # pair is one sample, so level counts follow from the bytes
            body = rows[:, 640:]
            n_hi = int((body.abs() > 2).sum().item())
            n_neg = int((body < 0).sum().item())
            assert abs(n_hi / body.numel() - 0.5) < 1e-3
            assert abs(n_neg / body.numel() - 0.5) < 1e-3
        del raw, back


def test_c4_full_32gib_guppi_stream():
    nchan, npol, spf, ov = 512, 2, 65536, 512
    fbytes = nchan * spf * npol * 2                  # 128 MiB per frame
    nfr = 8                                          # 1 GiB chunks
    off = torch.arange(nfr, dtype=torch.int64, device=DEV) * fbytes
    cb = torch.zeros(nfr, dtype=torch.int64, device=DEV)
    ce = torch.full((nfr,), spf * npol, dtype=torch.int64, device=DEV)
    oc0 = torch.arange(nfr, dtype=torch.int64, device=DEV) * (spf * npol)
    out = torch.empty((nfr * spf * npol * nchan * 2,), dtype=torch.float32,
                      device=DEV)
    g = torch.Generator(device=DEV).manual_seed(3000)
    for k in range(32):
        raw = torch.randint(0, 256, (nfr * fbytes,), dtype=torch.uint8,
                            device=DEV, generator=g)
        kernels.decode_int8_transposed(raw, off, nfr, nchan, spf * npol, 2,
                                       cb, ce, oc0, out)
        back = torch.zeros_like(raw)
        kernels.encode_int8_transposed(out, back, off, nfr, nchan,
                                       spf * npol, 2)
        assert torch.equal(back, raw), 'chunk %d' % k
        if k % 8 == 0:
            want = int(raw.view(torch.int8).sum(dtype=torch.int64).item())
            got = out.sum(dtype=torch.float64).item()
            assert got == want
            # overlap windows: frames after the first skip `ov` samples
            cb2 = torch.full((nfr,), ov * npol, dtype=torch.int64,
                             device=DEV)
            cb2[0] = 0
            oc2 = torch.cumsum(ce - cb2, 0) - (ce - cb2)
            n2 = int((ce - cb2).sum().item()) * nchan * 2
            part = torch.empty((n2,), dtype=torch.float32, device=DEV)
            kernels.decode_int8_transposed(raw, off, nfr, nchan, spf * npol,
                                           2, cb2, ce, oc2, part)
            full = out.view(nfr, spf * npol, nchan * 2)
            keep = torch.cat([full[0]] + [full[i, ov * npol:]
                                          for i in range(1, nfr)])
            assert torch.equal(part.view(-1, nchan * 2), keep)
            del part, keep
        del raw, back


def test_c5_full_16gib_mark5b_stream():
    nframe = (1 << 30) // 10016
    lv = levels.mark5b(2)
    out = torch.empty((nframe * 2500, 16), dtype=torch.float32, device=DEV)
    for k in range(16):
        raw, valid = synthetic.mark5b_stream_device(nframe, DEV,
                                                    seed=4000 + k)
        fields, uo = kernels.mark5b_scan(raw, nframe)
        kernels.decode_bitfield(raw, uo, nframe, 1, 10000, 2, 16, False,
                                kernels.CODEC_LEVELS, lv, -999.0, out=out)
        got_valid = fields[kernels.M5B_VALID].cpu().numpy().astype(bool)
        assert np.array_equal(got_valid, valid), 'chunk %d' % k
        per = out.view(nframe, -1)
        filled = (per == -999.).all(1).cpu().numpy()
        assert np.array_equal(filled, ~valid)
        back = raw.clone()
        back.view(nframe, 10016)[:, 16:] = 0
        kernels.encode_bitfield(out, back, torch.where(
            uo >= 0, uo, torch.arange(nframe, device=DEV) * 10016 + 16),
            nframe, 1, 10000, 2, 16, kernels.QUANT_MARK5B)
        ok = torch.from_numpy(valid).to(DEV)
        assert torch.equal(back.view(nframe, 10016)[ok],
                           raw.view(nframe, 10016)[ok]), 'chunk %d' % k
        del raw, back


def test_large_irregular_stream_index():
    """The GPU frame index at size: 256 MiB of VDIF frame sets in pinned host
    memory with 1 % of the frames dropped, some swapped and a few bytes cut
    out of one frame.  The table must be exactly what the damage implies, and
    a read through it must give fill_value for the lost frames and the
    reference decode (oracle) for sampled intact ones."""
    import time
    import warnings
    nthread, payload, frame = 8, 5000, 5032
    nset = (256 << 20) // (nthread * frame)
    raw = synthetic.vdif_stream(nset, nthread, payload, seed=12,
                                thread_order=np.arange(nthread))
    frames = raw.reshape(nset * nthread, frame)
    rng = np.random.default_rng(4)
    nframe = nset * nthread
    keep = np.ones(nframe, bool)
    keep[rng.choice(np.arange(nthread * 4, nframe - nthread * 4),
                    nframe // 100, replace=False)] = False
    order = np.flatnonzero(keep)
    for a in rng.choice(order.size - 2, 50, replace=False):
        order[[a, a + 1]] = order[[a + 1, a]]               # swapped pairs
    blob = frames[order].reshape(-1)
    cut_at = int(order.size // 2)                 # cut 3 bytes out of a frame
    cut = cut_at * frame + 1000
    blob = np.concatenate([blob[:cut], blob[cut + 3:]])
    lost_by_cut = int(order[cut_at])
    expect = np.full((nset, nthread), -1, np.int64)
    for pos, f in enumerate(order):
        if f == lost_by_cut:
            continue
        off = pos * frame - (3 if pos > cut_at else 0)
        s, t = divmod(int(f), nthread)
        expect[s, t] = off
    src = HostBuffer(blob)
    with warnings.catch_warnings(record=True):
        warnings.simplefilter('always')
        fh = bb.vdif.open(src, 'rs', sample_rate=40e6, fill_value=-5.,
                          device=DEV)
        if fh._index is None:
            fh.read(1)                            # detection during a read
        t0 = time.perf_counter()
        fh._build_index()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        print('index of %.0f MiB built in %.1f ms (%.1f GB/s)' % (
            blob.size / 2**20, dt * 1e3, blob.size / dt / 1e9))
        table = fh._index
        assert table.shape == expect.shape
        assert np.array_equal(table, expect)
        fh.seek(0)
        data = fh.read()
    assert tuple(data.shape) == (nset * 20000, nthread)
    gone = np.argwhere(expect < 0)
    assert len(gone) == nframe // 100 + 1
    for s, t in gone[:40]:
        assert bool((data[s * 20000:(s + 1) * 20000, t] == -5.).all())
    for s, t in rng.integers(0, [nset, nthread], (12, 2)):
        if expect[s, t] < 0:
            continue
        words = frames[s * nthread + t, 32:].view('<u4')
        want = codec.vdif_payload_decode(words, 2, (1,), False)[:, 0]
        got = data[s * 20000:(s + 1) * 20000, t].cpu().numpy()
        assert np.array_equal(got.view('u4'), want.view('u4'))
    fh.close()


def test_int8_moments_one_huge_unit():
    """bb_int8_moments over one 1.25 GiB unit: a single CTA-thread then sees
    more than 2^18 words, the point at which its 32-bit partial sums of
    squares must have been folded into the 64-bit totals.  Worst case first
    (every sample -128), then a period-4 pattern with known per-lane sums."""
    n = 5 << 28                                       # bytes, multiple of 16
    nword = n // 4
    uo = torch.zeros(1, dtype=torch.int64, device=DEV)
    raw = torch.full((n,), 0x80, dtype=torch.uint8, device=DEV)
    got = torch.zeros((1, 1, 4, 3), dtype=torch.int64, device=DEV)
    kernels.int8_moments(raw, uo, 1, 1, n, 4, got)
    want = np.array([[nword, -128 * nword, 16384 * nword]] * 4)
    assert np.array_equal(got.cpu().numpy()[0, 0], want)
    pattern = np.array([-128, 127, -1, 3], np.int8)
    raw.view(torch.int32).fill_(int(pattern.view(np.int32)[0]))
    got.zero_()
    kernels.int8_moments(raw, uo, 1, 1, n, 4, got)
    want = np.stack([np.full(4, nword), pattern.astype(np.int64) * nword,
                     pattern.astype(np.int64) ** 2 * nword], axis=1)
    assert np.array_equal(got.cpu().numpy()[0, 0], want)
    # one element (real, single polarisation): the four lanes are summed
    got1 = torch.zeros((1, 1, 1, 3), dtype=torch.int64, device=DEV)
    kernels.int8_moments(raw, uo, 1, 1, n, 1, got1)
    assert np.array_equal(got1.cpu().numpy()[0, 0, 0], want.sum(axis=0))


@pytest.mark.parametrize('payload,nset', [(128 << 10, 512), (8 << 20, 3)])
def test_state_counts_4bit_counter_limits(payload, nset):
    """4-bit state counts keep pairs of 16-bit counters per lane: one bin of
    512 units of 128 KiB makes the launcher split the bin so that no lane
    passes 2^16 words; 8 MiB units are beyond what one lane may take and go
    to the histogram kernel.  All nibbles are one element here, so numpy's
    bincount is the answer."""
    g = torch.Generator(device=DEV).manual_seed(payload % 1000 + nset)
    raw = torch.randint(0, 256, (nset * payload,), dtype=torch.uint8,
                        device=DEV, generator=g)
    uo = torch.arange(nset, dtype=torch.int64, device=DEV) * payload
    got = torch.zeros((1, 1, 1, 16), dtype=torch.int64, device=DEV)
    kernels.state_counts(raw, uo, nset, 1, payload, 4, 1, got)
    host = raw.cpu().numpy()
    want = np.bincount(host & 15, minlength=16) \
        + np.bincount(host >> 4, minlength=16)
    assert np.array_equal(got.cpu().numpy()[0, 0, 0], want)
    # two elements (a complex channel): low nibbles are re, high nibbles im
    got2 = torch.zeros((1, 1, 2, 16), dtype=torch.int64, device=DEV)
    kernels.state_counts(raw, uo, nset, 1, payload, 4, 2, got2)
    assert np.array_equal(got2.cpu().numpy()[0, 0, 0],
                          np.bincount(host & 15, minlength=16))
    assert np.array_equal(got2.cpu().numpy()[0, 0, 1],
                          np.bincount(host >> 4, minlength=16))


# ---------------------------------------------------------------------------
# Partial reads across a launch split.  The planner cuts a call whose item
# count would pass 32 bits (the warp-cooperative modes: 2^26 word positions)
# into several launches; every later one carries a shifted row base and unit
# offset pointer.  These cases read from inside a frame of the first launch
# to inside a frame of the last, with invalid units on both sides of the
# split, and check the sets next to the split and the partial end frames
# bit for bit against the oracle, the fill count of the whole range exactly,
# and the decode -> encode round trip of the whole range.
@pytest.fixture(scope='module')
def emu():
    import emu_build
    return emu_build.load()


def _frames(nunit, payload, seed):
    """nunit frames of a 32-byte header and `payload` random bytes."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    raw = torch.randint(0, 256, (nunit * (payload + 32),), dtype=torch.uint8,
                        device=DEV, generator=g)
    uo = torch.arange(nunit, dtype=torch.int64, device=DEV) * (payload + 32) \
        + 32
    return raw, uo


@pytest.mark.parametrize('mode,nthread,align', [('WORDRUN', 1, 4),
                                                ('WORDROW4', 4, 1)])
def test_partial_read_across_launch_split(emu, mode, nthread, align):
    from bitfield_cases import plan_decode
    bps, nelem, payload, fill = 8, 1, 8000, -999.0
    spf, frame = payload, payload + 32
    nset = 0x3ffffff // (payload // 4) + 7      # just past one launch
    start = (spf // 3) // align * align + align
    end = ((nset - 1) * spf + 2 * spf // 3) // align * align
    got_mode, _, nlaunch, split, _ = plan_decode(
        emu, nset, nthread, payload, bps, nelem, start, end - start)
    assert (got_mode, nlaunch) == (mode, 2) and 0 < split < nset - 1
    raw, uo = _frames(nset * nthread, payload, 77 + nthread)
    invalid = sorted({split * nthread - 1, split * nthread,
                      (split + 1) * nthread - 1})
    uo_inv = uo.clone()
    uo_inv[invalid] = -1
    lv = levels.offset_binary(8)
    out = kernels.decode_bitfield(raw, uo_inv, nset, nthread, payload, bps,
                                  nelem, False, kernels.CODEC_LEVELS, lv,
                                  fill, start, end - start)
    frames = raw.view(nset * nthread, frame)

    def want_set(s):
        rows = np.empty((spf, nthread), np.float32)
        for t in range(nthread):
            u = s * nthread + t
            rows[:, t] = fill if u in invalid else codec.vdif_decode(
                frames[u, 32:].cpu().numpy().view('<u4'), bps)
        return rows

    for s in (0, split - 1, split, nset - 1):
        lo, hi = max(s * spf, start), min((s + 1) * spf, end)
        want = want_set(s)[lo - s * spf:hi - s * spf]
        got = out[lo - start:hi - start, :, 0].cpu().numpy()
        assert np.array_equal(got.view('u4'), want.view('u4')), s
    nfill = sum(min((u // nthread + 1) * spf, end)
                - max(u // nthread * spf, start) for u in invalid)
    assert int((out == fill).sum().item()) == nfill
    del out
    # the whole range decoded and encoded back: the valid units' payloads
    full = kernels.decode_bitfield(raw, uo_inv, nset, nthread, payload, bps,
                                   nelem, False, kernels.CODEC_LEVELS, lv,
                                   fill)
    back = torch.zeros_like(raw)
    kernels.encode_bitfield(full, back, uo_inv, nset, nthread, payload, bps,
                            nelem, kernels.QUANT_OFFSET_BINARY)
    want = raw.clone()
    want.view(-1, frame)[:, :32] = 0
    want.view(-1, frame)[invalid] = 0
    assert torch.equal(back, want)


def test_rowword_encode_across_launch_split(emu):
    """2-bit, two complex threads (ROWWORD2): just over 2^26 word positions,
    invalid units on both sides of the split stay untouched, the valid ones
    re-encode to the payload they were decoded from."""
    from bitfield_cases import plan_encode
    bps, nelem, nthread, payload = 2, 2, 2, 8000
    frame = payload + 32
    nset = 0x3ffffff // (payload // 4) + 5
    mode, _, nlaunch, split, _ = plan_encode(emu, nset, nthread, payload,
                                             bps, nelem)
    assert (mode, nlaunch) == ('ROWWORD2', 2) and 0 < split < nset - 1
    raw, uo = _frames(nset * nthread, payload, 91)
    data = kernels.decode_bitfield(raw, uo, nset, nthread, payload, bps,
                                   nelem, True, kernels.CODEC_LEVELS,
                                   levels.offset_binary(2))
    invalid = [split * nthread - 2, split * nthread - 1, split * nthread + 1,
               nset * nthread - 1]
    uo_inv = uo.clone()
    uo_inv[invalid] = -1
    back = torch.full_like(raw, 0xEE)
    kernels.encode_bitfield(data, back, uo_inv, nset, nthread, payload, bps,
                            nelem, kernels.QUANT_OFFSET_BINARY)
    want = raw.clone()
    want.view(-1, frame)[:, :32] = 0xEE
    want.view(-1, frame)[invalid] = 0xEE
    assert torch.equal(back, want)
