"""8-bit state counts through the host layer on the CPU emulation backend,
with the numpy restatement of bb_byte_counts standing in for the kernel
(tests/byte_count_cases.py); the same cases run on the GPU in
tests/test_gpu_byte_counts.py."""
import numpy as np
import pytest
import torch

import byte_count_cases as cases


@pytest.fixture
def backend(monkeypatch):
    cases.install(monkeypatch)


@pytest.mark.parametrize('case', cases.CASES, ids=lambda f: f.__name__)
def test_case(backend, case):
    case()


def test_restatement_checks_table_shape():
    c = cases.kernel_case(np.random.default_rng(0), 4, 2, 'uniform')
    with pytest.raises(ValueError):
        cases.byte_counts(torch.from_numpy(c['raw']), torch.from_numpy(c['uo']),
                          c['nset'], 2, c['payload'], 4,
                          torch.zeros((9, 2, 4, 16), dtype=torch.int64))


def test_moments_unchanged_by_shared_view(backend):
    """tasks.moments goes through the shared unit-table helper: its shapes
    for every layout are those of the sample shape."""
    import baseband_b200 as bb
    from baseband_b200 import tasks
    from conftest import sample_path
    with bb.guppi.open(sample_path('sample_puppi.raw'), 'rs') as fh:
        n, total, sq = tasks.moments(fh)
        assert n.shape == (1,) + fh.sample_shape + (2,)


@pytest.mark.timeout(300)
def test_sharded_gloo():
    cases.run_sharded(use_cpu=True)
