"""Subset reads without a GPU: the selective decoders' bodies (CPU
emulation, tests/emu/emu_select.cpp) against numpy restatements, and every
format's reader with a ``subset`` on the CPU emulation backend
(tests/cpu_backend.py).  The same checks run on the B200 in
tests/test_gpu_subset.py."""
import pytest

import reduced_cases
import subset_cases


@pytest.fixture
def backend(monkeypatch):
    import cpu_backend
    cpu_backend.install(monkeypatch)


@pytest.mark.parametrize('case', subset_cases.bitfield_cases(),
                         ids=lambda c: 'bps{bps}-t{nthread}-e{nelem}'.format(
                             **c))
def test_select_bitfield(backend, case):
    subset_cases.check_bitfield(case, 'cpu')


def test_select_bitfield_wide_table(backend):
    subset_cases.check_bitfield_launch_split('cpu')


@pytest.mark.parametrize('case', subset_cases.int8_cases(),
                         ids=lambda c: '-'.join(map(str, c)))
def test_select_int8(backend, case):
    subset_cases.check_int8(case, 'cpu')


@pytest.mark.parametrize('name', sorted(reduced_cases.STREAMS))
def test_stream_subsets(backend, name):
    subset_cases.check_stream(name, 'cpu')


def test_ways_of_reading(backend):
    subset_cases.check_ways_of_reading('cpu')
