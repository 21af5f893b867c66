"""float16 / bfloat16 encoder input without a GPU: the encode kernels'
bodies at both 16-bit input types (tests/emu/emu_reduced_encode.cpp) and
the stream writers on the CPU emulation backend (tests/cpu_backend.py).  The
rule throughout: a 16-bit value encodes to exactly the bytes of its float32
value.  The same cases run on the B200 in tests/test_gpu_reduced_encode.py."""
import ctypes

import numpy as np
import pytest
import torch

import reduced_encode_cases as rec


@pytest.fixture
def backend(monkeypatch):
    import cpu_backend
    return cpu_backend.install(monkeypatch)


def test_host_widening_is_exact(backend):
    """The emulation's widening of every 16-bit pattern is the exact float32
    value (NaN with its sign)."""
    backend.emu_widen_half.restype = None
    backend.emu_widen_half.argtypes = [ctypes.c_void_p, ctypes.c_int64,
                                       ctypes.c_int32, ctypes.c_void_p]
    for dtype in rec.HALF:
        x = rec.all_patterns(dtype)
        bits = x.view(torch.int16).numpy().copy()
        out = np.empty(bits.size, np.float32)
        backend.emu_widen_half(ctypes.c_void_p(bits.ctypes.data), bits.size,
                               int(dtype == torch.bfloat16),
                               ctypes.c_void_p(out.ctypes.data))
        assert np.array_equal(out.view(np.uint32),
                              rec.widen(x).numpy().view(np.uint32))


@pytest.mark.parametrize('dtype', rec.HALF, ids=str)
def test_exhaustive_bitfield(backend, dtype):
    report = {}
    rec.exhaustive_bitfield('cpu', dtype, report)
    print('output bytes the float64 (numpy) encode changes:', report)


@pytest.mark.parametrize('dtype', rec.HALF, ids=str)
def test_exhaustive_mark4(backend, dtype):
    rec.exhaustive_mark4('cpu', dtype)


@pytest.mark.parametrize('dtype', rec.HALF, ids=str)
def test_exhaustive_int8(backend, dtype):
    rec.exhaustive_int8('cpu', dtype)


def test_matrix_cells(backend):
    """Every float32 encode cell of the planner (all kernel instances,
    partly filled last rounds, invalid units, special values)."""
    from bitfield_cases import matrix_cases
    cases = [c for c in matrix_cases()[1] if c['dtype'] == 'f4']
    assert len(cases) == 44
    for case in cases:
        rec.matrix_cell('cpu', case)


def test_alignment(backend):
    rec.check_alignment('cpu')


@pytest.mark.parametrize('name', rec.WRITER_STREAMS)
def test_writers(backend, name):
    rec.check_writer(name, 'cpu')


def test_type_errors(backend):
    rec.check_type_errors('cpu')


@pytest.mark.parametrize('name', rec.ROUND_TRIP_STREAMS)
def test_round_trip(backend, name):
    rec.check_round_trip(name, 'cpu')
