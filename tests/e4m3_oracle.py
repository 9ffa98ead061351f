"""Float64 restatement of the E4M3 storage rule of ``PackedCorpus(dtype="e4m3")`` (include/mfar_b200.h,
``mfar_corpus_pack_rows_e4m3``) - test infrastructure, the checker the pack kernel is compared with bit for bit.
It rounds once, from float64, by its own arithmetic (``np.rint`` on exactly scaled values), not through torch's cast."""
from __future__ import annotations

from typing import Tuple

import numpy as np
import torch

from mfar_oracle import NORM_EPS


E4M3_MAX = 448.0
E4M3_SCALE_EXP = (-117, 119)            # 2^-9 * 2^-117 = 2^-126 (normal fp32 / bf16); 448 * 2^119 finite in bf16


def e4m3_rne(v) -> np.ndarray:
    """float64 -> the nearest E4M3 value (ties to even), as float64: ONE rounding, subnormal spacing 2^-9, saturating
    to +-448.  Signs of zeros are kept."""
    v = np.asarray(v, dtype=np.float64)
    _, k = np.frexp(v)                                  # |v| = m 2^k, 0.5 <= m < 1: 4 significant bits -> 2^(k-4)
    q = np.maximum(k - 4, -9)
    r = np.ldexp(np.rint(np.ldexp(v, -q)), q)           # exact scalings; rint rounds half to even
    return np.clip(r, -E4M3_MAX, E4M3_MAX) + 0.0 * v    # + 0.0 * v keeps the sign of a zero result


def e4m3_bytes(vals) -> np.ndarray:
    """E4M3 values (float64, exactly representable) -> their uint8 encodings (sign | exponent 4 bits, bias 7 |
    mantissa 3 bits); a negative zero is 0x80."""
    vals = np.asarray(vals, dtype=np.float64)
    a = np.abs(vals)
    m, k = np.frexp(a)
    normal = a >= 2.0 ** -6
    b = np.where(normal, ((k + 6) << 3) | np.rint(m * 16 - 8).astype(np.int64), np.rint(a * 512).astype(np.int64))
    return (b | np.where(np.signbit(vals), 0x80, 0)).astype(np.uint8)


def quantize_rows_e4m3(x, normalize: bool = False) -> Tuple[np.ndarray, np.ndarray]:
    """The E4M3 storage rule of ``PackedCorpus(dtype="e4m3")`` for docs and queries alike.  Every row, taken exactly
    into float64 (and, with ``normalize``, divided by ``max(||x||_2, float32(1e-12))`` in float64), gets the scale
    s = 2^e, e = clamp(ceil(log2(amax / 448)), -117, 119), and the payload p = RNE_e4m3(x / s), rounded once.
    A row of zeros (either sign) stores s = 1 and payload 0; a row holding a NaN or an infinity s = NaN and payload 0.
    Returns (payload uint8 [n, d], scales float32 [n])."""
    if torch.is_tensor(x):
        x = x.detach().cpu().double().numpy()
    x = np.asarray(x, dtype=np.float64)
    bad = ~np.all(np.isfinite(x), axis=1)
    xf = np.where(bad[:, None], 0.0, x)
    if normalize:
        norm = np.sqrt(np.sum(xf * xf, axis=1, keepdims=True))
        xf = xf / np.maximum(norm, NORM_EPS)
    amax = np.max(np.abs(xf), axis=1) if xf.shape[1] else np.zeros(xf.shape[0])
    m, k = np.frexp(amax)
    e = np.clip(k - 9 + (m > 0.875), *E4M3_SCALE_EXP)   # the least e with amax <= 448 * 2^e
    zero = (amax == 0) | bad
    e = np.where(zero, 0, e)
    payload = e4m3_bytes(e4m3_rne(np.ldexp(xf, -e[:, None])))
    payload[zero] = 0
    scales = np.where(bad, np.nan, np.ldexp(1.0, e)).astype(np.float32)
    return payload, scales


def dequantize_rows_e4m3(payload: np.ndarray, scales: np.ndarray) -> np.ndarray:
    """float32 [n, d] = E4M3 value of each byte * the row's scale (exact: every product is a normal fp32 number)."""
    b = np.asarray(payload, dtype=np.uint8).astype(np.int64)
    e, mant = (b >> 3) & 15, b & 7
    mag = np.where(e == 0, mant * 2.0 ** -9, (1 + mant / 8.0) * np.ldexp(1.0, e - 7))
    val = np.where(b & 0x80, -mag, mag)
    return (val.astype(np.float32) * np.asarray(scales, dtype=np.float32)[:, None]).astype(np.float32)
