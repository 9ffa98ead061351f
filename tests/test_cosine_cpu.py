"""The cosine contract of the reference (``mfar_oracle.normalize_rows_bf16``) on values worked out by hand.

Every row, taken exactly into float64, is divided by max(||x||_2, float32(1e-12)) and rounded ONCE to nearest-even bf16.
The expected values below are either literal or computed with exact rational arithmetic (``fractions``), so the
helper is checked against something that shares none of its float64 steps.
"""
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

import mfar_oracle as O

EPS = Fraction(float(np.float32(1e-12)))


def rne_fraction(f: Fraction) -> Fraction:
    """Exact nearest-even bf16 of a rational: 8 significant bits, subnormal spacing 2^-133."""
    if f == 0:
        return Fraction(0)
    a = abs(f)
    e = math.floor(math.log2(a))                      # 2^e <= a < 2^(e+1), then correct the float log
    while Fraction(2) ** e > a:
        e -= 1
    while Fraction(2) ** (e + 1) <= a:
        e += 1
    q = Fraction(2) ** max(e - 7, -133)
    n = a / q
    lo = math.floor(n)
    rem = n - lo
    m = lo + (1 if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and lo % 2) else 0)
    return (m * q) if f > 0 else -(m * q)


def exact_row(row):
    """The contract in rationals: the norm is irrational in general, so bracket it tightly enough to decide."""
    xs = [Fraction(float(v)) for v in row]
    ss = sum(v * v for v in xs)
    out = []
    # sqrt(ss) to ~2^-200 relative by integer square root of a scaled sum (the rounding boundaries are far coarser)
    scale = 2 ** 400
    s_int = ss * scale * scale
    r = math.isqrt(s_int.numerator // s_int.denominator)
    norm = max(Fraction(r, scale), EPS)
    for v in xs:
        out.append(rne_fraction(v / norm))
    return out


def sums_of_squares(total):
    """Greedy integers whose squares add up to ``total`` exactly."""
    out = []
    while total:
        r = math.isqrt(total)
        out.append(r)
        total -= r * r
    return out


def helper(rows, dtype=np.float32):
    return O.normalize_rows_bf16(np.asarray(rows, dtype=dtype))


def bits(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(torch.bfloat16).view(torch.int16)


def test_round_bf16_rne_midpoints_both_ways():
    u = 2.0 ** -8                                          # half of the bf16 spacing at 1.0
    y = np.array([1 + u, 1 + 3 * u, -(1 + u), -(1 + 3 * u), 1 + u * (1 + 2 ** -30), 1 + u * (1 - 2 ** -30),
                  2.0 ** 127 * (2 - 2 ** -8), 2.0 ** 127 * (2 - 2 ** -7)])
    want = np.array([1.0, 1 + 4 * u, -1.0, -(1 + 4 * u), 1 + 2 * u, 1.0, np.inf, 2.0 ** 127 * (2 - 2 ** -7)])
    assert np.array_equal(O.round_bf16_rne(y), want)


def test_round_bf16_rne_subnormals_and_zero_signs():
    s = 2.0 ** -133                                        # bf16 subnormal spacing
    y = np.array([0.5 * s, 1.5 * s, 2.5 * s, 0.49 * s, 127.5 * s, 2.0 ** -126 - 0.5 * s, -1.5 * s, 0.0, -0.0,
                  -0.25 * s])
    got = O.round_bf16_rne(y)
    want = np.array([0.0, 2 * s, 2 * s, 0.0, 128 * s, 2.0 ** -126, -2 * s, 0.0, -0.0, -0.0])
    assert np.array_equal(got, want)
    assert np.array_equal(np.signbit(got), np.signbit(want))
    assert np.array_equal(bits(got), bits(want))


def test_normalized_midpoints_round_half_even():
    """257/512 and 259/512 are exact bf16 midpoints: rows with those quotients and an integer norm of 512."""
    rows = []
    for lead in (257, 259, -257, -259):
        rest = sums_of_squares(512 * 512 - lead * lead)
        rows.append([lead] + rest + [0] * (8 - len(rest)))
    got = helper(rows)
    assert got[0, 0] == 0.5 and got[1, 0] == 260 / 512 and got[2, 0] == -0.5 and got[3, 0] == -260 / 512
    for row, g in zip(rows, got):
        assert [Fraction(float(v)) for v in g] == exact_row(row)


def test_norms_either_side_of_eps():
    e = float(np.float32(1e-12))
    t_lo, t_hi = 2.0 ** -43, 2.0 ** -42                  # 5 t is below eps for t_lo, above it for t_hi
    rows = [[e / 2, 0.0], [e, 0.0], [2 * e, 0.0], [e / 2, e / 2], [3 * t_lo, 4 * t_lo], [3 * t_hi, 4 * t_hi],
            [-e / 4, 0.0]]
    got = helper(rows)
    assert got[0].tolist() == [0.5, 0.0] and got[1].tolist() == [1.0, 0.0] and got[2].tolist() == [1.0, 0.0]
    assert got[3].tolist() == [0.5, 0.5] and got[6].tolist() == [-0.25, 0.0]
    assert got[5].tolist() == [0.6015625, 0.80078125]     # bf16(0.6), bf16(0.8): the norm 5 t_hi is used
    assert got[4, 0] < 0.6 and got[4, 1] < 0.8             # below eps the row is divided by eps, not by its norm
    for row, g in zip(rows, got):
        assert [Fraction(float(v)) for v in g] == exact_row(row)


def test_zero_rows_and_signs_of_zero():
    rows = np.array([[0.0, -0.0, 0.0, -0.0], [-0.0] * 4, [0.0] * 4, [-0.0, 3.0, -0.0, -4.0]], dtype=np.float32)
    got = helper(rows)
    assert np.array_equal(bits(got), bits(np.array([[0.0, -0.0, 0.0, -0.0], [-0.0] * 4, [0.0] * 4,
                                                     [-0.0, 0.6015625, -0.0, -0.80078125]], dtype=np.float32)))


def test_single_nonzero_is_exactly_one():
    vals = [1.0, -1.0, 3.0, 1e-11, -(2.0 ** 120), 1e30, 2.0 ** -39]      # every |x| above eps
    rows = np.zeros((len(vals), 5), dtype=np.float32)
    rows[np.arange(len(vals)), np.arange(len(vals)) % 5] = vals
    got = helper(rows)
    assert np.array_equal(got.sum(axis=1), np.sign(vals))
    assert (np.count_nonzero(got, axis=1) == 1).all()


def test_rows_above_2_pow_64():
    rows = [[2.0 ** 70, 0.0, 0.0, 0.0], [3 * 2.0 ** 80, -4 * 2.0 ** 80, 0, 0], [2.0 ** 100] * 4,
            [2.0 ** 126, 2.0 ** 126, 2.0 ** 126, -(2.0 ** 126)], [1.8e19, 1.8e19, 1.8e19, 1.8e19]]
    got = helper(rows)
    assert got[0].tolist() == [1.0, 0.0, 0.0, 0.0]
    assert got[1].tolist() == [0.6015625, -0.80078125, 0.0, 0.0]
    assert got[2].tolist() == [0.5] * 4 and got[3].tolist() == [0.5, 0.5, 0.5, -0.5] and got[4].tolist() == [0.5] * 4


def test_tiny_components_land_on_bf16_subnormals():
    s = 2.0 ** -133
    rows = [[1.0, 3 * 2.0 ** -134], [1.0, 5 * 2.0 ** -135], [1.0, 2.0 ** -130], [1.0, 2.0 ** -135]]
    got = helper(rows)
    # the float64 norm of each row is exactly 1 (the tiny square is far below its ulp), so 1.5 * 2^-133 is a tie that
    # goes to the even 2^-132, 1.25 * 2^-133 rounds down and 0.25 * 2^-133 flushes to +0
    assert got[:, 0].tolist() == [1.0] * 4
    assert got[:, 1].tolist() == [2 * s, s, 8 * s, 0.0]


def test_bf16_and_f16_sources_are_taken_exactly():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(64, 100, generator=g)
    for dt in (torch.bfloat16, torch.float16):
        xd = x.to(dt)
        assert np.array_equal(O.normalize_rows_bf16(xd), O.normalize_rows_bf16(xd.float().numpy()))


@pytest.mark.parametrize("scale", [1.0, 1e-6, 1e15, 2.0 ** -60])   # fp32 squares stay finite and normal
def test_agrees_with_torch_normalize_away_from_midpoints(scale):
    """fp32 ``F.normalize`` then bf16 rounds twice; away from a bf16 midpoint (2^-20 relative) both must agree."""
    g = torch.Generator().manual_seed(7)
    mu = torch.randn(768, generator=g)
    x = (torch.randn(2000, 768, generator=g) + 0.5 * mu) * scale
    ours = O.normalize_rows_bf16(x)
    theirs = torch.nn.functional.normalize(x, dim=1).to(torch.bfloat16).float().numpy()
    xd = x.double().numpy()
    y = xd / np.maximum(np.sqrt((xd * xd).sum(axis=1, keepdims=True)), O.NORM_EPS)
    safe = O.round_bf16_rne(y * (1 + 2.0 ** -20)) == O.round_bf16_rne(y * (1 - 2.0 ** -20))
    assert safe.mean() > 0.999
    assert np.array_equal(ours[safe], theirs[safe])
    assert np.array_equal(ours, O.round_bf16_rne(y))


def test_exhaustive_scores_normalize_path():
    g = torch.Generator().manual_seed(5)
    fields = [torch.randn(50, 64, generator=g) * 3 for _ in range(2)]
    q = torch.randn(4, 64, generator=g)
    w = torch.full((1, 2), 0.5)
    got = O.exhaustive_scores(q, fields, None, w, normalize=True)
    qn = torch.from_numpy(O.normalize_rows_bf16(q))
    want = 0.5 * (qn @ torch.from_numpy(O.normalize_rows_bf16(fields[0])).T) + \
        0.5 * (qn @ torch.from_numpy(O.normalize_rows_bf16(fields[1])).T)
    torch.testing.assert_close(got, want, rtol=1e-6, atol=1e-7)
    assert not torch.allclose(got, O.exhaustive_scores(q, fields, None, w))
