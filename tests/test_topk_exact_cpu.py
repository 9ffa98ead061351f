"""The premise of tests/test_gpu_topk_exact.py, checked without a GPU: the closed-form scores and top-k of every
(pattern, sign) equal a float64 brute force over the doc matrix the GPU tests pack, and every score stays in the range
where any summation order is exact in fp32.  A failure here is a broken test input, not a kernel bug."""
import numpy as np
import pytest

import exact_topk as X


@pytest.mark.parametrize("N", [129, 4097, 9001])
@pytest.mark.parametrize("dim", [64, 768])
def test_closed_form_matches_float64_brute_force(N, dim):
    docs = X.doc_matrix(N, dim).astype(np.float64)
    n = np.arange(N)
    for name, sign in X.COMBOS:
        q = X.query_vector(name, sign, dim).astype(np.float64)
        s64 = docs @ q
        want = X.dense_scores(name, sign, N)
        assert np.array_equal(s64, want.astype(np.float64)), (name, sign)
        # every partial sum of the products is an integer of magnitude < 2^24: exact in fp32 in any order
        assert (np.abs(docs * q).sum(axis=1) < 2 ** 24).all(), (name, sign)
        # fp32 in two different orders gives the same integers
        d32, q32 = docs.astype(np.float32), q.astype(np.float32)
        assert np.array_equal((d32 * q32).sum(axis=1, dtype=np.float32), want.astype(np.float32))
        assert np.array_equal((d32[:, ::-1] * q32[::-1]).cumsum(axis=1, dtype=np.float32)[:, -1], want.astype(np.float32))
        for k in (1, 2, 100, 127, 128):
            ref = np.lexsort((n, -s64))[:k]
            assert np.array_equal(X.topk_order(want, k), ref), (name, sign, k)


def test_patterns_put_ties_at_rank_k():
    """The tie patterns really tie at rank k (else they would test nothing) and the controls really do not."""
    N = 4097
    for name, sign in X.COMBOS:
        s = X.dense_scores(name, sign, N)
        kth = s[X.topk_order(s, 100)[-1]]
        tied = int((s == kth).sum())
        if name in ("n", "perm"):
            assert tied == 1, name
        elif name != "planted" or sign < 0:
            assert tied > 1, (name, sign)
    assert (X.dense_scores("planted", 1, N) > 0).sum() < 100          # fewer than k winners above the tied floor


def test_query_coefficients_and_coordinates_exact_in_bf16():
    torch = pytest.importorskip("torch")
    for name, sign in X.COMBOS:
        q = torch.from_numpy(X.query_vector(name, sign, 768))
        assert torch.equal(q.to(torch.bfloat16).float(), q)
    d = torch.from_numpy(X.doc_matrix(4097, 768).astype(np.float32))
    assert torch.equal(d.to(torch.bfloat16).float(), d)
