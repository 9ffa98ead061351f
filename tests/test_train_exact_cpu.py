"""The premises of tests/test_gpu_train_exact.py, checked without a GPU.  A failure here is a broken test input or a
bound that is too tight, not a kernel bug.

- Every field-component case: the float64 reference equals an integer brute force that addresses doc n = p*Neg + s
  itself, every output's sum of |terms| is below 2^24 (so every partial sum is exact in fp32, whatever the order and
  however the bwd_q slices split the N*F rows), and fp32 in two different orders gives the same values.
- Every mixture case: torch CPU fp32 (the oracle, with autograd) stays inside the per-element bound
  ``exact_train.mixture_bounds``."""
import numpy as np
import pytest
import torch

import exact_train as X
import train_oracle as T


def test_case_table_covers_every_axis_value():
    cs = X.COMPONENT_CASES
    assert {c.B for c in cs} >= set(X._BS) and {c.E for c in cs} >= set(X._ES) and {c.F for c in cs} >= set(X._FS)
    assert {c.Neg for c in cs} >= set(X._NEGS) and {c.grads for c in cs} == set(X._GRADS)
    assert {c.dtype for c in cs} == set(X.DTYPES) and {c.T for c in cs} == set(X._TS)
    rows = {c.rows for c in cs}
    assert {1, 15, 16, 17, 4736, 4737} <= rows and max(rows) >= 50000
    assert 60 <= len(cs) <= 100 and len(set(map(X.case_id, cs))) == len(cs)
    ms = X.MIXTURE_CASES
    assert {c[0] for c in ms} == set(X._MIX_FS) and {c[1] for c in ms} == set(X._MIX_SS)
    assert {c[2] for c in ms} == set(X._MIX_BS) and {c[3] for c in ms} == set(X._MIX_ES)
    assert {c[4] for c in ms} == {True, False} and {c[5] for c in ms} == set(X._SUBSETS)


def _brute_force(q, docs, G, T):
    """int64 contraction with the doc index decoded by hand (n -> p = n // Neg, s = n % Neg)."""
    qi, di, Gi = (t.numpy().astype(np.int64) for t in (q, docs, G))
    B, E = qi.shape
    if di.ndim == 3:
        nfe = di
    else:
        P, F, Neg, _ = di.shape
        nfe = np.stack([di[n // Neg, :, n % Neg, :] for n in range(P * Neg)])
    N, F, _ = nfe.shape
    D = nfe.reshape(N * F, E)
    comp = (qi @ D.T).reshape(B, N, F)
    dq = Gi.reshape(B, N * F) @ D
    dd = (Gi.reshape(B, N * F).T @ qi).reshape(N, F, E)
    if di.ndim == 4:
        dd = dd.reshape(P, Neg, F, E).transpose(0, 2, 1, 3)
    return [torch.from_numpy(np.ascontiguousarray(a)).double() / T for a in (comp, dq, dd)]


@pytest.mark.parametrize("case", X.COMPONENT_CASES, ids=X.case_id)
def test_component_references_are_exact(case):
    q, docs, G = X.component_inputs(case)
    assert q.abs().max() <= 3 and docs.abs().max() <= 3 and G.abs().max() <= 2
    assert (G != 0).any()
    ref = X.components_reference(q, docs, G, case.T)
    for a, b in zip(ref, _brute_force(q, docs, G, case.T)):
        assert torch.equal(a, b)
    # every partial sum of every output is a multiple of 1/T below 2^24 in magnitude: exact in fp32
    for mag in X.components_magnitudes(q, docs, G, case.T):
        assert float(mag.max()) < 2 ** 24
    # fp32 in two different summation orders (the contraction axis reversed) gives the reference
    q32, d32, G32 = q.float(), X.docs_as_nfe(docs).float(), G.float()
    N, F, E = d32.shape
    D = d32.reshape(N * F, E)
    for rev in (False, True):
        qq, DD, GG = (q32.flip(1), D.flip(1), G32.flip(1)) if rev else (q32, D, G32)
        GG2 = G32.reshape(case.B, N * F)
        comp = (qq @ DD.t()).reshape(case.B, N, F) / case.T
        dq = ((GG2.flip(1) @ D.flip(0)) if rev else (GG2 @ D)) / case.T
        dd = ((GG2.t().flip(1) @ q32.flip(0)) if rev else (GG2.t() @ q32)) / case.T
        assert torch.equal(comp.double(), ref[0])
        assert torch.equal(dq.double(), ref[1])
        assert torch.equal(dd.reshape(N, F, E).double(), X.docs_as_nfe(ref[2]))


def _cpu_fp32_mixture(x, q, W, qc, g):
    x, q, W = (t.clone().requires_grad_(True) for t in (x, q, W))
    out = T.mixture(x, q, W, qc)
    (out * g).sum().backward()
    r = {"out": out.detach(), "dx": x.grad, "dW": W.grad}
    if qc:
        r["dq"] = q.grad
        r["w"] = torch.softmax(q.detach() @ W.detach(), dim=1)
    else:
        r["w"] = torch.softmax(W.detach().t(), dim=1)
    return r


@pytest.mark.parametrize("case", X.MIXTURE_CASES, ids=X.mixture_case_id)
def test_mixture_bound_holds_for_torch_cpu_fp32(case):
    F, S, B, E, qc, _ = case
    x, q, W, g = X.mixture_inputs(B, S, F, E, qc, seed=F * 100 + S + B + E)
    ref = X.mixture_reference(x, q, W, qc, g)
    bound = X.mixture_bounds(x, q, W, qc, g)
    got = _cpu_fp32_mixture(x, q, W, qc, g)
    for k in ("w", "out", "dW") + (("dq",) if qc else ()):
        err = (got[k].double() - ref[k]).abs()
        assert (err <= bound[k]).all(), (k, float((err / bound[k]).max()))
    # the logits really are spread, and the bound stays below the weight's own size on the tiny weights too (unless
    # the weight under-flows)
    assert float(ref["logits"].max() - ref["logits"].min()) >= (20 if F > 2 else 0)
    assert ((bound["w"] < 0.25 * ref["w"]) | (ref["w"] < 2.0 ** -100)).all()


def test_mixture_bound_rejects_a_wrong_small_weight():
    """A relative error of 1e-3 on a weight of about 1e-18 is outside the bound (query_cond False: exact logits)."""
    x, q, W, g = X.mixture_inputs(3, 37, 7, 4, False, seed=5)
    W = torch.tensor([[0.0], [-20.7], [1.0], [-3.0], [2.0], [-40.0], [0.5]])
    ref = X.mixture_reference(x, q, W, False, g)
    bound = X.mixture_bounds(x, q, W, False, g)
    w = float(ref["w"][0, 5])
    assert 1e-19 < w < 1e-17
    assert w * 1e-3 > float(bound["w"][0, 5])


def test_row_bar_sees_a_wrong_small_row():
    """The loss bar is per element: a row 2^16 smaller than its neighbour, off by 1 %, fails it."""
    f64 = torch.stack([torch.full((8,), 1.0), torch.full((8,), 2.0 ** -16)]).double()
    cpu32 = f64.float()
    bar = X.row_bar(cpu32, f64)
    wrong = f64.clone()
    wrong[1] *= 1.01
    assert ((wrong - f64).abs() > bar).any()
    assert ((f64.float().double() - f64).abs() <= bar).all()
