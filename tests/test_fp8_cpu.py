"""The E4M3 storage rule of ``PackedCorpus(dtype="e4m3")`` as the oracle states it (``e4m3_oracle.quantize_rows_e4m3``),
checked without a GPU: against torch's own float8_e4m3fn cast wherever the two rules coincide, at the scale clamps, on
zero / non-finite / saturating rows and after the cosine normalisation."""
import numpy as np
import pytest
import torch

import e4m3_oracle as E
import mfar_oracle as O


def _torch_bytes(x: np.ndarray, scales: np.ndarray) -> np.ndarray:
    """torch's fp32 -> float8_e4m3fn cast (round to nearest even) of x / s.  x / s is exact in fp32 here (s is a power
    of two and the quotient stays normal), so the cast rounds once, as the oracle does from float64."""
    q = torch.from_numpy((x.astype(np.float64) / scales[:, None].astype(np.float64)).astype(np.float32))
    return q.to(torch.float8_e4m3fn).view(torch.uint8).numpy()


def test_every_e4m3_value_round_trips():
    b = np.arange(256, dtype=np.uint8)
    b = b[(b & 0x7F) != 0x7F]                               # 0x7F / 0xFF are NaN
    ref = torch.from_numpy(b.copy()).view(torch.float8_e4m3fn).float().numpy().astype(np.float64)
    vals = E.dequantize_rows_e4m3(b[None, :], np.ones(1, np.float32))[0]
    assert np.array_equal(vals.view(np.uint32), ref.astype(np.float32).view(np.uint32))
    assert np.array_equal(E.e4m3_bytes(E.e4m3_rne(ref)), b)


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("spread", [1e-3, 1.0, 1e6])
def test_random_rows_match_torch_cast(seed, spread):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((500, 96)) * spread * np.exp(rng.uniform(-8, 8, (500, 1)))).astype(np.float32)
    x[:, ::7] *= np.float32(1e-5)                          # subnormal E4M3 payloads
    p, s = E.quantize_rows_e4m3(x)
    assert np.array_equal(p, _torch_bytes(x, s))
    assert np.all(np.abs(x).max(axis=1) <= 448 * s.astype(np.float64))
    assert np.all(np.abs(x).max(axis=1) > 224 * s.astype(np.float64))          # e is the least such exponent


def test_ties_round_to_even():
    # 1.0625 lies halfway between 1.0 and 1.125: to 1.0 (even mantissa); 1.1875 halfway between 1.125 and 1.25: to 1.25
    x = np.array([[448.0, 1.0625, 1.1875, -1.0625, 2.0 ** -10, 3 * 2.0 ** -10, -(2.0 ** -11)]], dtype=np.float32)
    p, s = E.quantize_rows_e4m3(x)
    assert s[0] == 1.0
    d = E.dequantize_rows_e4m3(p, s)[0]
    assert d.tolist() == [448.0, 1.0, 1.25, -1.0, 0.0, 2.0 ** -8, -0.0]
    assert p[0, 6] == 0x80                                   # a negative value that rounds to zero keeps its sign
    assert np.array_equal(p, _torch_bytes(x, s))


def test_scale_clamps_and_saturation():
    big = np.float32(1.75 * 2.0 ** 127)
    x = np.array([[2.0 ** -140, 0.0],                       # e would be -148: clamped to -117, payload underflows to 0
                  [2.0 ** -120, 2.0 ** -125],               # e = -117 keeps 2^-9 * 2^-117 = 2^-126
                  [big, 1.0],                               # e = 119, exactly 448 * 2^119
                  [np.float32(3.3e38), -np.float32(3.3e38)]],  # past 448 * 2^119: saturates to +-448
                 dtype=np.float32)
    p, s = E.quantize_rows_e4m3(x)
    assert s.tolist() == [2.0 ** -117, 2.0 ** -117, 2.0 ** 119, 2.0 ** 119]
    d = E.dequantize_rows_e4m3(p, s)
    assert d[0].tolist() == [0.0, 0.0]
    assert d[1, 0] == 2.0 ** -120 and d[1, 1] == 2.0 ** -125    # payload 2^-8: a subnormal E4M3, a normal bf16
    assert d[2, 0] == big
    assert p[3].tolist() == [0x7E, 0xFE] and d[3].tolist() == [float(448 * 2.0 ** 119), -float(448 * 2.0 ** 119)]


def test_zero_and_non_finite_rows():
    x = np.array([[0.0, -0.0, 0.0], [1.0, np.nan, 2.0], [np.inf, 1.0, 1.0], [-np.inf, 0.0, 0.0], [-0.0, -0.0, -0.0]],
                 dtype=np.float32)
    for normalize in (False, True):
        p, s = E.quantize_rows_e4m3(x, normalize=normalize)
        assert not p.any()
        assert s[0] == 1.0 and s[4] == 1.0 and np.isnan(s[1:4]).all()
        d = E.dequantize_rows_e4m3(p, s)
        assert (d[[0, 4]] == 0).all() and np.isnan(d[1:4]).all()


def test_normalize_then_quantize_rounds_once_from_float64():
    rng = np.random.default_rng(5)
    x = rng.standard_normal((300, 64)).astype(np.float32)
    x[0] = 0.0
    x[1] = np.float32(1e-30) * x[1]                          # norm below eps: divided by 1e-12, not by the norm
    x[2, :] = 0.0; x[2, 5] = -3.0                            # one non-zero element: exactly -1
    x[3] = np.float32(1e19) * x[3]                           # squares overflow fp32, not float64
    p, s = E.quantize_rows_e4m3(x, normalize=True)
    y = x.astype(np.float64)
    y = y / np.maximum(np.sqrt((y * y).sum(1, keepdims=True)), O.NORM_EPS)
    assert np.array_equal(E.dequantize_rows_e4m3(p, s).astype(np.float64),
                          E.e4m3_rne(np.ldexp(y, -np.log2(s.astype(np.float64)).astype(int)[:, None]))
                          * s.astype(np.float64)[:, None])
    assert s[0] == 1.0 and not p[0].any()
    assert E.dequantize_rows_e4m3(p[2:3], s[2:3])[0, 5] == -1.0
    assert np.all(np.abs(E.dequantize_rows_e4m3(p[3:4], s[3:4])) <= 1.0)


def test_dequantized_values_are_bf16_numbers():
    rng = np.random.default_rng(9)
    x = (rng.standard_normal((400, 128)) * np.exp(rng.uniform(-80, 80, (400, 1)))).astype(np.float32)
    for normalize in (False, True):
        p, s = E.quantize_rows_e4m3(x, normalize=normalize)
        d = E.dequantize_rows_e4m3(p, s)
        rt = torch.from_numpy(d).to(torch.bfloat16).float().numpy()
        assert np.array_equal(rt.view(np.uint32), d.view(np.uint32))
        nz = d[d != 0]
        assert np.all(np.abs(nz) >= np.float32(2.0 ** -126))          # normal: never a subnormal fp32 / bf16
