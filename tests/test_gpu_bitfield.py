"""GPU parity: the CUDA bit-field kernels, called through the C ABI, against
the oracle on the shared case table, the reference golden vectors and
size-independent properties at larger sizes."""
import numpy as np
import pytest
import torch

from baseband_b200 import kernels, levels
from oracle import codec
from bitfield_cases import (DECODE_CASES, ENCODE_CASES, make_decode_case,
                            oracle_decode, make_encode_case, oracle_encode,
                            matrix_cases)

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


MATRIX_DECODE, MATRIX_ENCODE = matrix_cases()
# floats of sentinel on either side of a decode's output (64 KiB each; a
# multiple of four floats keeps the output 16-byte aligned)
GUARD = 16384
SENTINEL = 0x7FBADBAD               # a NaN payload no decode produces


@pytest.mark.parametrize('case', DECODE_CASES + MATRIX_DECODE,
                         ids=lambda c: c['id'])
def test_decode_bitfield(case):
    """Decode into a view of a larger buffer: the values must equal the
    oracle bit for bit and the sentinels around the view stay untouched."""
    c = make_decode_case(case)
    want = oracle_decode(c)
    buf = torch.full((want.size + 2 * GUARD,), SENTINEL, dtype=torch.int32,
                     device=DEV).view(torch.float32)
    view = buf[GUARD:GUARD + want.size].view(want.shape)
    out = kernels.decode_bitfield(
        _t(c['raw']), _t(c['unit_offset']), c['nset'], c['nthread'],
        c['payload_nbytes'], c['bps'], c['nelem'], c['complex'], c['codec'],
        c['levels'], c['fill'], c['sample_start'], c['nsample'], out=view)
    assert out.data_ptr() == view.data_ptr()
    got = buf.cpu().numpy().view('u4')
    assert np.array_equal(got[GUARD:GUARD + want.size], want.ravel().view('u4'))
    assert (got[:GUARD] == SENTINEL).all() and (got[-GUARD:] == SENTINEL).all()


@pytest.mark.parametrize('case', ENCODE_CASES + MATRIX_ENCODE,
                         ids=lambda c: c['id'])
def test_encode_bitfield(case):
    c = make_encode_case(case)
    want = oracle_encode(c)
    dst = torch.full((c['dst_nbytes'],), 0xEE, dtype=torch.uint8, device=DEV)
    kernels.encode_bitfield(_t(c['data']), dst, _t(c['unit_offset']),
                            c['nset'], c['nthread'], c['payload_nbytes'],
                            c['bps'], c['nelem'], c['quantiser'])
    assert np.array_equal(dst.cpu().numpy(), want)


def test_golden_codec_vectors(codec_vectors):
    g = codec_vectors
    words = _t(g['words32'].view(np.uint8))
    off = torch.zeros(1, dtype=torch.int64, device=DEV)
    nb = g['words32'].nbytes
    for key, bps, codec_id, lv in (
            ('vdif_dec1', 1, 0, levels.offset_binary(1)),
            ('vdif_dec2', 2, 0, levels.offset_binary(2)),
            ('vdif_dec4', 4, 0, levels.offset_binary(4)),
            ('vdif_dec8', 8, 0, levels.offset_binary(8)),
            ('m5b_dec1', 1, 0, levels.mark5b(1)),
            ('m5b_dec2', 2, 0, levels.mark5b(2))):
        out = kernels.decode_bitfield(words, off, 1, 1, nb, bps, 1, False,
                                      codec_id, lv)
        assert np.array_equal(out.cpu().numpy().ravel().view('u4'),
                              g[key].view('u4')), key
    b = _t(g['bytes'].view(np.uint8))
    for key, bps in (('gsb4_dec', 4), ('int8_dec', 8)):
        out = kernels.decode_bitfield(b, off, 1, 1, g['bytes'].nbytes, bps,
                                      1, False, kernels.CODEC_SINT)
        assert np.array_equal(out.cpu().numpy().ravel(), g[key]), key
    for tag in ('f32', 'f64'):
        vals, finite = _t(g['enc_in_' + tag]), _t(g['enc_in_finite_' + tag])
        for quant, name, bpss, src in (
                (0, 'vdif_enc%d_', (1, 2, 4, 8), vals),
                (1, 'm5b_enc%d_', (1, 2), vals),
                (2, {4: 'gsb4_enc_', 8: 'int8_enc_'}, (4, 8), finite)):
            for bps in bpss:
                key = (name[bps] if isinstance(name, dict)
                       else name % bps) + tag
                want = g[key]
                dst = torch.zeros(want.size, dtype=torch.uint8, device=DEV)
                kernels.encode_bitfield(src, dst, off, 1, 1, want.size, bps,
                                        1, quant)
                bad = np.nonzero(dst.cpu().numpy() != want)[0]
                assert bad.size == 0, (key, bad[:5])


def test_nan_encode(codec_vectors):
    g = codec_vectors
    nanv = _t(g['nan_in'])
    off = torch.zeros(1, dtype=torch.int64, device=DEV)
    for key, bps, quant in (('vdif_enc2_nan', 2, 0), ('vdif_enc1_nan', 1, 0),
                            ('m5b_enc1_nan', 1, 1)):
        want = g[key]
        dst = torch.zeros(want.size, dtype=torch.uint8, device=DEV)
        kernels.encode_bitfield(nanv, dst, off, 1, 1, want.size, bps, 1,
                                quant)
        assert np.array_equal(dst.cpu().numpy(), want), key


@pytest.mark.parametrize('bps,nthread,nelem', [(2, 16, 1), (2, 1, 16),
                                               (1, 8, 1), (4, 2, 2),
                                               (8, 4, 8)])
def test_large_round_trip(bps, nthread, nelem):
    """encode(decode(x)) == x on 64 MiB of random payload (every code is a
    fixed point of decode->encode), plus a sampled oracle comparison."""
    payload = 8000
    nset = (64 << 20) // (payload * nthread)
    g = torch.Generator(device=DEV).manual_seed(1234)
    raw = torch.randint(0, 256, (nset * nthread * payload,),
                        dtype=torch.uint8, device=DEV, generator=g)
    off = torch.arange(nset * nthread, dtype=torch.int64, device=DEV) * payload
    lv = levels.offset_binary(bps)
    out = kernels.decode_bitfield(raw, off, nset, nthread, payload, bps,
                                  nelem, False, 0, lv)
    back = torch.zeros_like(raw)
    kernels.encode_bitfield(out, back, off, nset, nthread, payload, bps,
                            nelem, 0)
    assert torch.equal(back, raw)
    # float64 input encodes to the same codes
    if bps == 2:
        back64 = torch.zeros_like(raw[:payload * nthread * 4])
        kernels.encode_bitfield(out[:4 * (payload * 8 // (bps * nelem))]
                                .double().contiguous(), back64,
                                off[:4 * nthread], 4, nthread, payload, bps,
                                nelem, 0)
        assert torch.equal(back64, raw[:payload * nthread * 4])
    # sampled units against the oracle
    spf = payload * 8 // (bps * nelem)
    host = out.cpu().numpy()
    rawh = raw.cpu().numpy()
    rng = np.random.default_rng(5)
    for u in rng.integers(0, nset * nthread, 16):
        s, t = divmod(int(u), nthread)
        want = codec.vdif_decode(rawh[u * payload:(u + 1) * payload]
                                 .view('<u4'), bps).reshape(spf, nelem)
        assert np.array_equal(host[s * spf:(s + 1) * spf, t], want)


def test_errors():
    raw = torch.zeros(64, dtype=torch.uint8, device=DEV)
    off = torch.zeros(1, dtype=torch.int64, device=DEV)
    with pytest.raises(KeyError):     # no 3-bit decoder
        kernels.decode_bitfield(raw, off, 1, 1, 64, 2, 1, False, 1, None)
    with pytest.raises(ValueError):
        kernels.decode_bitfield(raw, off, 1, 1, 62, 2, 1, False, 0,
                                levels.offset_binary(2))
    with pytest.raises(TypeError):    # no CPU fallback
        kernels.decode_bitfield(raw.cpu(), off, 1, 1, 64, 2, 1, False, 0,
                                levels.offset_binary(2))


def test_fuzz_bitfield():
    """400 seeded random geometries (all planner modes, partial ranges,
    invalid units, both float widths) through the C ABI vs the oracle."""
    from bitfield_cases import fuzz_cases
    dec, enc = fuzz_cases(400, seed=20260102)
    for case in dec:
        test_decode_bitfield(case)
    for case in enc:
        test_encode_bitfield(case)
