"""Subset reads on the B200: the selective decoders against numpy
restatements, every format's reader with a ``subset`` against the full read
indexed (tests/subset_cases.py, also run on the CPU emulation by
tests/test_host_subset.py), and the device memory a subset read takes."""
import numpy as np
import pytest
import torch

import baseband_b200 as bb
from baseband_b200 import synthetic
from baseband_b200.base.memory import HostBuffer
import reduced_cases
import subset_cases

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.mark.parametrize('case', subset_cases.bitfield_cases(),
                         ids=lambda c: 'bps{bps}-t{nthread}-e{nelem}'.format(
                             **c))
def test_select_bitfield(case):
    subset_cases.check_bitfield(case, DEV)


def test_select_bitfield_wide_table():
    subset_cases.check_bitfield_launch_split(DEV)


@pytest.mark.parametrize('case', subset_cases.int8_cases(),
                         ids=lambda c: '-'.join(map(str, c)))
def test_select_int8(case):
    subset_cases.check_int8(case, DEV)


@pytest.mark.parametrize('name', sorted(reduced_cases.STREAMS))
def test_stream_subsets(name):
    subset_cases.check_stream(name, DEV)


def test_ways_of_reading():
    subset_cases.check_ways_of_reading(DEV)


def _growth(read):
    """Peak device memory ``read()`` allocates beyond what was held."""
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    result = read()
    torch.cuda.synchronize()
    return result, torch.cuda.max_memory_allocated() - before


def test_guppi_subset_memory():
    """C4 channel geometry (512 channels x 2 pol, complex int8): a device
    read of one channel of one polarisation allocates its own width, not the
    8 KiB per sample of a full decode (1 GiB here)."""
    nframe, spf = 32, 4096
    raw, data = synthetic.guppi_stream(nframe, nchan=512, npol=2,
                                       samples_per_frame=spf, overlap=0,
                                       seed=9)
    full_nbytes = nframe * spf * 512 * 2 * 2 * 4
    assert full_nbytes >= 1 << 30
    with bb.guppi.open(HostBuffer(raw), 'rs', device=DEV,
                       subset=(0, 7)) as fh:
        got, grown = _growth(fh.read)
    assert grown < full_nbytes // 4, grown
    want = data[7, :, 0].astype(np.float32).view(np.complex64)[:, 0]
    subset_cases.same(got, torch.from_numpy(want))


def test_mark4_subset_memory():
    """A Mark 4 subset is gathered chunk by chunk from the stage's scratch:
    the read allocates the selected width, not the whole decoded rows."""
    h0 = bb.mark4.Mark4Header.fromvalues(
        64, time='2014-06-16T07:38:12.475', bps=2, fanout=4, nsb=1)
    nframe = 420                       # 33.6 M samples x 8 channels
    lv = torch.tensor([-3.316505, -1., 1., 3.316505], device=DEV)
    g = torch.Generator(device=DEV).manual_seed(4)
    sink = HostBuffer(nframe * 160000)
    fw = bb.mark4.open(sink, 'ws', header0=h0, sample_rate=32e6, device=DEV)
    for k in range(0, nframe, 60):
        n = min(60, nframe - k) * 80000
        fw.write(lv[torch.randint(0, 4, (n, 8), device=DEV, generator=g)])
    fw._flush(final=False)
    del fw
    torch.cuda.empty_cache()
    full_nbytes = nframe * 80000 * 8 * 4
    assert full_nbytes >= 1 << 30
    opts = dict(ntrack=64, decade=2010, device=DEV, chunk_nbytes=1 << 20)
    # (closing a reader closes the buffer: the reference is read first)
    ref = bb.mark4.open(sink, 'rs', **opts)
    ref.seek(123457)
    want = ref.read(1000000)[:, 5]
    with bb.mark4.open(sink, 'rs', subset=5, **opts) as fh:
        got, grown = _growth(fh.read)
    assert grown < full_nbytes // 4, grown
    subset_cases.same(got[123457:1123457], want)

