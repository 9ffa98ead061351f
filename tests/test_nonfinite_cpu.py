"""The top-k rule for NaN and infinite scores on the CPU side: the oracle's ranking (``mfar_oracle.rank_rows`` /
``topk_sorted``), the host key packing (``dist.encode_keys``) and the closed-form inputs of tests/exact_nonfinite.py.

Rule: NaN (any sign or payload, one value) > +inf > finite scores descending > -inf; the lower row first in a class.
"""
import numpy as np
import pytest
import torch

import exact_nonfinite as NF
import exact_topk as X
import mfar_oracle as O


def _nan(bits):
    return np.array([bits], dtype=np.uint32).view(np.float32)[0]


NANS = [np.float32(np.nan), -np.float32(np.nan), _nan(0x7F800001), _nan(0xFFC00001), _nan(0xFFFFFFFF)]


def _row(rng, N, p_nan, p_inf, n_levels):
    """fp32 row with ties (n_levels distinct finite values), +-0.0, NaNs of every sign and payload, +-inf."""
    x = rng.integers(-n_levels, n_levels + 1, N).astype(np.float32) * np.float32(0.25)
    x[rng.random(N) < 0.05] = -0.0
    u = rng.random(N)
    x[u < p_inf] = np.inf
    x[(u >= p_inf) & (u < 2 * p_inf)] = -np.inf
    nan_at = np.nonzero(rng.random(N) < p_nan)[0]
    x[nan_at] = np.array(NANS, dtype=np.float32)[rng.integers(0, len(NANS), nan_at.size)]
    return x


@pytest.mark.parametrize("seed", range(12))
def test_rank_rows_matches_brute_force(seed):
    rng = np.random.default_rng(seed)
    N = int(rng.integers(1, 700))
    p_nan, p_inf = [(0.0, 0.0), (0.02, 0.02), (0.3, 0.2), (0.9, 0.0), (0.0, 0.45)][seed % 5]
    x = _row(rng, N, p_nan, p_inf, int(rng.integers(1, 50)))
    for k in (1, 7, 100, 128, N):
        want = NF.brute_force_order(x, k)
        got = O.rank_rows(x, k)
        assert np.array_equal(got, want), f"N={N} k={k}"
    s, i = O.topk_sorted(torch.from_numpy(np.stack([x, x[::-1].copy()])), 100)
    assert np.array_equal(i[0].numpy(), NF.brute_force_order(x, 100))
    assert np.array_equal(i[1].numpy(), NF.brute_force_order(x[::-1], 100))
    assert np.array_equal(np.isnan(s[0].numpy()), np.isnan(x[i[0].numpy()]))


@pytest.mark.parametrize("seed", range(6))
def test_rank_rows_matches_torch_topk_without_ties(seed):
    """Tie-free rows (distinct finite values, at most one NaN, +inf and -inf, the NaN of either sign): the same ids as
    torch.topk, which is what the reference ranks with (contrastive.py:696)."""
    rng = np.random.default_rng(100 + seed)
    N = 300
    x = rng.permutation(N).astype(np.float32) - 150.0
    special = rng.choice(N, 3, replace=False)
    x[special] = [NANS[seed % len(NANS)], np.inf, -np.inf]
    for k in (1, 2, 3, 50, N):
        want = torch.topk(torch.from_numpy(x), k).indices.numpy()
        assert np.array_equal(O.rank_rows(x, k), want), f"k={k}"


def test_encode_keys_folds_every_nan_above_inf():
    from mfar_b200.dist import decode_keys, encode_keys
    vals = np.array(NANS + [np.inf, np.float32(3.0e38), 1.0, 0.0, -1.0, -np.inf], dtype=np.float32)
    ids = np.arange(vals.size, dtype=np.int64) + 7
    keys = encode_keys(vals, ids)
    words = keys >> np.uint64(32)
    assert (words[:len(NANS)] == np.uint64(0xFFC00000)).all()
    assert np.array_equal(words, O.ordered_words(vals))
    assert (np.diff(words[len(NANS) - 1:].astype(np.int64)) < 0).all(), "NaN > +inf > finite desc > -inf"
    s, i = decode_keys(keys)
    assert np.isnan(s[:len(NANS)]).all() and np.array_equal(s[len(NANS):], vals[len(NANS):])
    assert np.array_equal(i, ids)
    # one class: the lower id wins whichever NaN it holds
    order = np.argsort(keys[:len(NANS)])[::-1]
    assert np.array_equal(order, np.arange(len(NANS)))


@pytest.mark.parametrize("N,dim", [(4097, 768), (4097, 64), (330_001, 768)])
def test_planted_inputs_closed_form(N, dim):
    """The planted coordinates are free of pattern groups, the plant sets have the sizes the GPU tests rely on, and
    ``dense_values`` equals an element-wise IEEE evaluation of the bf16 doc rows times the query (on a doc sample)."""
    S = NF.plant_sets(N)
    assert S["few"].sum() < 100 and S["many"].sum() > 128 and (~S["almost"]).sum() < 60
    assert S["many"][:148 * 128].sum() >= 128                          # >= k inside the seeding prefix
    pos = NF.reserved(dim)
    used = set()
    for g in range(len(X.GROUPS)):
        used |= set(X.group_positions(g, dim))
    assert not used & set(pos.values())
    rows = np.unique(np.r_[np.nonzero(S["nan"] | S["few"])[0], np.arange(0, N, max(1, N // 300))])
    docs = X.doc_matrix(N, dim)[rows].astype(np.float64)
    for almost in (False, True):
        cols = NF.plant_columns(N, dim, almost)
        d = docs.copy()
        for p, bits in cols.items():
            b = bits[rows].view(np.uint16).astype(np.uint32) << 16
            with np.errstate(invalid="ignore"):
                v = b.view(np.float32).astype(np.float64)
            d[:, p] = np.where(bits[rows] != 0, v, d[:, p])
        assert np.isnan(d[S["nan"][rows], pos["nan"]]).all()
        nb = cols[pos["nan"]][rows][S["nan"][rows]].view(np.uint16)
        assert (nb & 0x8000).any() and (~nb & 0x8000).any(), "NaNs of both signs are planted"
        coefs_list = [c + (a,) for c in NF.COEFS for a in (1, -1, 0)] if almost else NF.COEFS
        for j, coefs in enumerate(coefs_list):
            combo = X.COMBOS[j % len(X.COMBOS)]
            q = NF.query_vector(combo, coefs, dim).astype(np.float64)
            with np.errstate(invalid="ignore"):
                want = (d * q[None, :]).sum(axis=1)
            got = NF.dense_values(combo, coefs, N, almost)[rows]
            assert np.array_equal(NF.classes(got), NF.classes(want))
            fin = NF.classes(want) == 1
            assert np.array_equal(got[fin], want[fin])
