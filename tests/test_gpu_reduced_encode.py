"""float16 / bfloat16 encoder input on the B200: the cases of
tests/test_host_reduced_encode.py against the CUDA library, and one 16-bit
encode across a launch split.  A 16-bit value must encode to exactly the
bytes of its float32 value."""
import pytest
import torch

import reduced_encode_cases as rec
from baseband_b200 import kernels, levels

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.mark.parametrize('dtype', rec.HALF, ids=str)
def test_exhaustive_bitfield(dtype):
    report = {}
    rec.exhaustive_bitfield(DEV, dtype, report)
    print('output bytes the float64 (numpy) encode changes:', report)


@pytest.mark.parametrize('dtype', rec.HALF, ids=str)
def test_exhaustive_mark4(dtype):
    rec.exhaustive_mark4(DEV, dtype)


@pytest.mark.parametrize('dtype', rec.HALF, ids=str)
def test_exhaustive_int8(dtype):
    rec.exhaustive_int8(DEV, dtype)


def test_matrix_cells():
    from bitfield_cases import matrix_cases
    cases = [c for c in matrix_cases()[1] if c['dtype'] == 'f4']
    assert len(cases) == 44
    for case in cases:
        rec.matrix_cell(DEV, case)


def test_alignment():
    rec.check_alignment(DEV)


@pytest.mark.parametrize('name', rec.WRITER_STREAMS)
def test_writers(name):
    rec.check_writer(name, DEV)


def test_type_errors():
    rec.check_type_errors(DEV)


@pytest.mark.parametrize('name', rec.ROUND_TRIP_STREAMS)
def test_round_trip(name):
    rec.check_round_trip(name, DEV)


@pytest.mark.parametrize('dtype', rec.HALF, ids=str)
def test_rowword_encode_across_launch_split(dtype):
    """2-bit, two complex threads (ROWWORD2) from 16-bit input: just over
    2^26 word positions, invalid units on both sides of the split stay
    untouched, the valid ones re-encode to the payload their samples were
    decoded from (every 2-bit level is exact at both 16-bit types)."""
    import emu_build
    from bitfield_cases import plan_encode
    emu = emu_build.load()
    bps, nelem, nthread, payload = 2, 2, 2, 8000
    frame = payload + 32
    nset = 0x3ffffff // (payload // 4) + 5
    mode, _, nlaunch, split, _ = plan_encode(emu, nset, nthread, payload,
                                             bps, nelem)
    assert (mode, nlaunch) == ('ROWWORD2', 2) and 0 < split < nset - 1
    gen = torch.Generator(device=DEV).manual_seed(93)
    raw = torch.randint(0, 256, (nset * nthread * frame,), dtype=torch.uint8,
                        device=DEV, generator=gen)
    uo = (torch.arange(nset * nthread, dtype=torch.int64, device=DEV) * frame
          + 32)
    data = kernels.decode_bitfield(raw, uo, nset, nthread, payload, bps,
                                   nelem, True, kernels.CODEC_LEVELS,
                                   levels.offset_binary(2), dtype=dtype)
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
