"""bb_byte_counts (csrc/bb_counts.cu) against its numpy restatement
(tests/byte_count_cases.py) through the C ABI -- every element window and
replica layout, shuffled / invalid / unaligned units, bins cutting the call,
accumulation, narrow and wide byte distributions, single units spread over
many CTAs, int64 totals past 2**32 -- and the 8-bit tasks.state_counts cases
on the GPU."""
import numpy as np
import pytest
import torch

import byte_count_cases as cases
from baseband_b200 import kernels

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'

NELEM = (1, 2, 4, 8, 16, 32, 64, 128, 256, 1024, 2048, 8192)
DISTS = ('uniform', 'one', 'two', 'narrow')


def _check(c):
    """One call equals the restatement, a second one adds as much again
    (compared on the device: no copies of the table beyond `want`)."""
    want = cases.kernel_want(c).to(DEV)
    got = torch.zeros(c['shape'], dtype=torch.int64, device=DEV)
    d_raw = torch.from_numpy(c['raw']).to(DEV)
    d_uo = torch.from_numpy(c['uo']).to(DEV)
    for _ in range(2):
        kernels.byte_counts(d_raw, d_uo, c['nset'], c['nthread'],
                            c['payload'], c['nelem'], got, c['origin'],
                            c['per_bin'])
        assert torch.equal(got, want), (c['nelem'], c['nthread'])
        got.sub_(want)


@pytest.mark.parametrize('nelem', NELEM)
def test_byte_counts_fuzz(nelem):
    """Every window / replica layout (they depend on nelem alone).  Threads
    x elements stay <= 8192, so that a table holds at most 16 MiB a bin:
    many threads are run with few elements."""
    rng = np.random.default_rng(7000 + nelem)
    for nthread in (n for n in (1, 2, 3, 16, 512) if n * nelem <= 8192):
        for dist in DISTS:
            unit = None
            if nthread == 512 or nelem >= 1024:
                # a few samples per unit: the restatement stays quick
                unit = nelem * int(rng.integers(1, 4)) * max(1, 4 // nelem)
            elif dist == 'narrow' and nthread == 1:
                unit = 512                       # MWA-sized payloads
            c = cases.kernel_case(rng, nelem, nthread, dist, unit_bytes=unit,
                                  nset=2 if nthread == 512 else None)
            assert np.prod(c['shape']) * 8 <= 6 * 16 * 2**20, c['shape']
            _check(c)


@pytest.mark.parametrize('nelem', (4, 2048))
def test_byte_counts_lone_unit(nelem):
    """One large unit per call (a DADA chunk piece): its segments are dealt
    out over many CTAs, 16-byte aligned or not."""
    rng = np.random.default_rng(90 + nelem)
    for dist in ('uniform', 'narrow'):
        c = cases.kernel_case(rng, nelem, 1, dist, nset=1,
                              unit_bytes=12 * 2**20)
        c['uo'] = np.abs(c['uo']) if c['uo'][0] >= 0 else np.array([4])
        _check(c)


def test_byte_counts_many_units():
    """Many small units over many CTAs per bin (the split), 16 threads."""
    rng = np.random.default_rng(5)
    for dist in DISTS:
        c = cases.kernel_case(rng, 2, 16, dist, nset=700, unit_bytes=512)
        c['per_bin'] = 300
        c['origin'] = 0
        c['shape'] = (3, 16, 2, 256)
        _check(c)


def test_byte_counts_errors():
    c = cases.kernel_case(np.random.default_rng(1), 4, 2, "uniform", nset=3)
    d_raw = torch.from_numpy(c['raw']).to(DEV)
    d_uo = torch.from_numpy(c['uo']).to(DEV)
    nbin = c['shape'][0]
    with pytest.raises(ValueError):                      # nelem not 2**k
        kernels.byte_counts(d_raw, d_uo, 1, 1, 12, 3, torch.zeros(
            (1, 1, 3, 256), dtype=torch.int64, device=DEV))
    with pytest.raises(ValueError):                      # table shape
        kernels.byte_counts(d_raw, d_uo, c['nset'], 2, c['payload'], 4,
                            torch.zeros((nbin, 2, 4, 16), dtype=torch.int64,
                                        device=DEV))
    with pytest.raises(ValueError):                      # past the last bin
        kernels.byte_counts(d_raw, d_uo, c['nset'], 2, c['payload'], 4,
                            torch.zeros((1, 2, 4, 256), dtype=torch.int64,
                                        device=DEV), 0, 1)
    with pytest.raises(ValueError):                      # misaligned src
        kernels.byte_counts(d_raw[1:], d_uo, 1, 1, 16, 4, torch.zeros(
            (1, 1, 4, 256), dtype=torch.int64, device=DEV))
    with pytest.raises(ValueError):                      # payload % nelem
        kernels.byte_counts(d_raw, d_uo, 1, 1, 24, 16, torch.zeros(
            (1, 1, 16, 256), dtype=torch.int64, device=DEV))


def test_byte_counts_past_2_32():
    """One unit of more than 4 GiB, every byte the same: the count is exact
    past 2**32 in the int64 table.  The unit's segments are spread over many
    CTAs.  That no CTA's 32-bit counters can wrap rests on the launcher
    giving none more than 2 GiB; driving one counter to 2**32 would take
    some 128 GiB through one CTA, more than a test can afford."""
    n = (1 << 32) + (1 << 28) + 4096
    raw = torch.full((n + 16,), 0x7d, dtype=torch.uint8, device=DEV)
    uo = torch.tensor([16], dtype=torch.int64, device=DEV)
    got = torch.zeros((1, 1, 1, 256), dtype=torch.int64, device=DEV)
    kernels.byte_counts(raw, uo, 1, 1, n, 1, got)
    got = got.cpu()
    assert got[0, 0, 0, 0x7d].item() == n
    assert got.sum().item() == n
    del raw
    torch.cuda.empty_cache()


@pytest.mark.parametrize('case', cases.CASES, ids=lambda f: f.__name__)
def test_stream_case(case):
    case()


@pytest.mark.timeout(300)
def test_sharded_gloo():
    cases.run_sharded(use_cpu=False)
