"""The training-time scorer (csrc/train.cu and the mixture kernels of csrc/aux_kernels.cu, through
``mfar_b200.modeling.losses`` / ``weighting``) element by element, at every tile and field edge.

1. Field components, forward and both gradients, on integer inputs where fp32 is exact in any order: compared with
   the float64 contraction by ``torch.equal`` (case table: tests/exact_train.py), plus the C ABI's refusals.
2. The field mixture, forward and backward, against float64 under the per-element bound
   ``exact_train.mixture_bounds``; dx = g * w bit for bit.
3. The contrastive losses at training sizes: loss and every gradient within 4 |cpu_fp32 - f64| + 2^-20 (row max) of
   float64, per element, with doc rows whose magnitudes span 2^-8 .. 2^8 (cpu_fp32: the larger deviation of two CPU
   summation orders).
4. [S,F] mixtures under autograd (the trec_eval_step form) keep their gradients."""
import copy
import math

import numpy as np
import pytest
import torch

import exact_train as X
import train_oracle as T

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _mods():
    from mfar_b200.modeling import losses as L
    from mfar_b200.modeling.weighting import LinearWeights
    return L, LinearWeights


def make_layer(W, query_cond):
    _, LinearWeights = _mods()
    layer = LinearWeights(W.shape[0], W.shape[1], query_cond=query_cond)
    with torch.no_grad():
        layer.weight.copy_(W)
    return layer.to(DEV)


def within(got, ref, bound, what):
    err = (got.detach().double() - ref.to(got.device).double()).abs()
    bound = bound.to(got.device)
    bad = ~(err <= bound)
    if bad.any():
        i = int(torch.argmax((err / bound).reshape(-1)))
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements outside the bound; worst at flat "
                             f"{i}: got {got.reshape(-1)[i].item():.9g}, f64 {ref.reshape(-1)[i].item():.9g}, "
                             f"bound {bound.reshape(-1)[i].item():.3g}")


# ---------------------------------------------------------------------------------------------------------------------
# 1. Field components: exact
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", X.COMPONENT_CASES, ids=X.case_id)
def test_field_components_exact(case):
    L, _ = _mods()
    dt = X.DTYPES[case.dtype]
    q64, d64, G64 = X.component_inputs(case, DEV)
    comp_ref, dq_ref, dd_ref = X.components_reference(q64, d64, G64, case.T)
    q = q64.to(dt).requires_grad_(case.grads in ("q", "both"))
    d = d64.to(dt).requires_grad_(case.grads in ("d", "both"))
    comp = L.field_components(q, d, case.T)
    assert comp.dtype == torch.float32 and comp.shape == (case.B, case.N, case.F)
    assert torch.equal(comp, comp_ref.float())
    comp.backward(G64.float())
    if q.requires_grad:
        assert q.grad.dtype == dt and torch.equal(q.grad, dq_ref.to(dt))
    else:
        assert q.grad is None
    if d.requires_grad:
        assert d.grad.dtype == dt and torch.equal(d.grad, dd_ref.to(dt))
    else:
        assert d.grad is None


def test_field_components_abi_refuses_inputs_outside_the_contract():
    """E % 4 != 0, E > 1024, F > 64 and a 4-byte-aligned (not 16-byte-aligned) view raise; nothing is written."""
    L, _ = _mods()
    from mfar_b200 import _native as nv
    for B, P, F, E in ((4, 3, 2, 6), (4, 3, 2, 1028), (4, 3, 65, 8)):
        with pytest.raises(RuntimeError):
            L.field_components(torch.ones(B, E, device=DEV), torch.ones(P, F, E, device=DEV), 1.0)
    P, F, E = 3, 2, 8
    buf = torch.ones(1 + P * F * E, device=DEV)
    docs = buf[1:].view(P, F, E)
    assert docs.is_contiguous() and docs.data_ptr() % 16 == 4
    with pytest.raises(RuntimeError):
        L.field_components(torch.ones(4, E, device=DEV), docs, 1.0)
    qbuf = torch.ones(1 + 4 * E, device=DEV)
    with pytest.raises(RuntimeError):
        L.field_components(qbuf[1:].view(4, E), torch.ones(P, F, E, device=DEV), 1.0)
    # the backward entry point: misaligned docs, dq or ddocs return an error before any launch
    q = torch.ones(4, E, device=DEV)
    good = torch.ones(P, F, E, device=DEV)
    g = torch.ones(4, P, F, device=DEV)
    dq_buf, dd_buf, dq_ok = (torch.full((n,), float("nan"), device=DEV) for n in (1 + 4 * E, 1 + P * F * E, 4 * E))
    for dq, dd, dc, out in ((dq_buf[1:], None, good, dq_buf), (None, dd_buf[1:], good, dd_buf),
                            (dq_ok, None, docs, dq_ok)):
        rc = nv.lib().mfar_field_components_bwd(nv.ptr(q), 4, E, nv.ptr(dc), P, F, 1, F * E, E, 0, 1.0, nv.ptr(g),
                                                nv.ptr(dq), nv.ptr(dd), nv.stream())
        torch.cuda.synchronize()
        assert rc != 0 and torch.isnan(out).all()


def test_decomposed_wrappers_exact_including_negatives():
    """compute_query_doc_field_components with Neg = 3 (doc order p*Neg + s) and compute_doc_query_scores against
    train_oracle in float64; W = 0 over F = 4 fields makes every mixture weight exactly 1/4."""
    L, _ = _mods()
    B, P, F, Neg, E, temp = 33, 5, 4, 3, 132, 0.5
    g = torch.Generator().manual_seed(7)
    q = torch.randint(-3, 4, (B, E), generator=g).double().to(DEV)
    dp = torch.randint(-3, 4, (P, F, E), generator=g).double().to(DEV)
    dn = torch.randint(-3, 4, (P, F, Neg, E), generator=g).double().to(DEV)
    W = torch.zeros(E, F, dtype=torch.float64)
    layer = make_layer(W.float(), True)
    mod = L.DecomposedContrastiveLoss(temperature=temp, all_gather_multi_gpu=False, mixture_of_fields_layer=layer)
    pc, nc = mod.compute_query_doc_field_components(q.float(), dp.float(), dn.float())
    rp, rn = T.field_components(q, dp, dn, temp)
    assert torch.equal(pc, rp.float()) and torch.equal(nc, rn.float())
    rev = mod.compute_doc_query_scores(dp.float(), q.float())
    assert torch.equal(rev, T.mixture(rp, q, W.to(DEV), True).t().float())


# ---------------------------------------------------------------------------------------------------------------------
# 2. Field mixture: per-element bounds
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", X.MIXTURE_CASES, ids=X.mixture_case_id)
def test_mixture_forward_backward_within_bound(case):
    F, S, B, E, qc, req = case
    x, q, W, g = X.mixture_inputs(B, S, F, E, qc, seed=F * 100 + S + B + E)
    ref = X.mixture_reference(x, q, W, qc, g)
    bound = X.mixture_bounds(x, q, W, qc, g)
    layer = make_layer(W, qc)
    layer.weight.requires_grad_("W" in req)
    xd = x.to(DEV).requires_grad_("x" in req)
    qd = q.to(DEV).requires_grad_("q" in req)
    out = layer(xd, qd if qc else None)
    within(out, ref["out"], bound["out"], "out")
    w = layer.field_weights(qd if qc else None)
    within(w, ref["w"], bound["w"], "weights")
    gd = g.to(DEV)
    if out.requires_grad:
        out.backward(gd)
    if "x" in req:
        assert torch.equal(xd.grad, gd[:, :, None] * w[:, None, :])           # one rounding of g * w ([1,F] static)
    else:
        assert xd.grad is None
    if "q" in req and qc:
        within(qd.grad, ref["dq"], bound["dq"], "dq")
    else:
        assert qd.grad is None
    if "W" in req and out.requires_grad:
        within(layer.weight.grad, ref["dW"], bound["dW"], "dW")
    else:
        assert layer.weight.grad is None


@pytest.mark.parametrize("F", [3, 33, 64])
def test_mixture_dx_is_one_row_of_weights_without_query_cond(F):
    """query_cond False: every b uses the same weight row, so dx / g is the same for every b, bit for bit."""
    B, S = 5, 37
    x, q, W, _ = X.mixture_inputs(B, S, F, 4, False, seed=F)
    g = torch.ones(B, S)
    layer = make_layer(W, False)
    xd = x.to(DEV).requires_grad_(True)
    layer(xd, None).backward(g.to(DEV))
    assert torch.equal(xd.grad, xd.grad[:1].expand_as(xd.grad))
    assert torch.equal(xd.grad[0, 0], layer.field_weights(None)[0])


@pytest.mark.parametrize("F", [2, 33, 64])
@pytest.mark.parametrize("qc", [True, False], ids=["qc", "static"])
def test_inference_weights_with_mask_and_two_dim_x(F, qc):
    """field_weights with a 0/1 mask (masked fields exactly 0) and the no-grad [S,F] x against B queries."""
    B, S, E = 5, 37, 100
    x, q, W, _ = X.mixture_inputs(B, S, F, E, qc, seed=3 * F)
    ref = X.mixture_reference(x, q, W, qc, torch.zeros(B, S))
    bound = X.mixture_bounds(x, q, W, qc, torch.zeros(B, S))
    layer = make_layer(W, qc)
    qd = q.to(DEV) if qc else None
    mask = (torch.arange(F) % 3 != 1).float()
    wm = layer.field_weights(qd, mask.to(DEV))
    within(wm, ref["w"] * mask, bound["w"] * mask, "masked weights")
    assert (wm[:, mask == 0] == 0).all()
    x2 = x[0]
    with torch.no_grad():
        out = layer(x2.to(DEV), qd)
    Bw = B if qc else 1
    r2 = X.mixture_reference(x2.expand(Bw, S, F), q, W, qc, torch.zeros(Bw, S))
    b2 = X.mixture_bounds(x2.expand(Bw, S, F), q, W, qc, torch.zeros(Bw, S))
    assert out.shape == (Bw, S)
    within(out, r2["out"], b2["out"], "[S,F] out")


# ---------------------------------------------------------------------------------------------------------------------
# 4. [S,F] x under autograd (weighting.py: the reference broadcasts [S,F] against [B,F] weights, differentiably)
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("qc", [True, False], ids=["qc", "static"])
def test_two_dim_x_keeps_its_gradients(qc):
    B, S, F, E = 5, 37, 7, 100
    x, q, W, _ = X.mixture_inputs(B, S, F, E, qc, seed=11)
    x2 = x[0]
    Bw = B if qc else 1
    g = torch.randn(Bw, S, generator=torch.Generator().manual_seed(12))
    layer = make_layer(W, qc)
    xd = x2.to(DEV).requires_grad_(True)
    qd = q.to(DEV).requires_grad_(True)
    out = layer(xd, qd if qc else None)
    assert out.shape == (Bw, S) and out.grad_fn is not None
    out.backward(g.to(DEV))
    x3 = x2.expand(Bw, S, F)
    ref = X.mixture_reference(x3, q, W, qc, g)
    bound = X.mixture_bounds(x3, q, W, qc, g)
    within(out, ref["out"], bound["out"], "out")
    # dx[s,f] = sum_b g[b,s] w[b,f]: exact terms summed over B by the expand's backward
    w = ref["w"].expand(Bw, F)
    dw = bound["w"].expand(Bw, F)
    ag = g.double().abs()
    dx_bound = ag.t() @ dw + X.gamma(Bw) * (ag.t() @ (w + dw)) + X.TINY
    within(xd.grad, ref["dx"].sum(0), dx_bound, "dx")
    within(layer.weight.grad, ref["dW"], bound["dW"], "dW")
    if qc:
        within(qd.grad, ref["dq"], bound["dq"], "dq")
    else:
        assert qd.grad is None


# ---------------------------------------------------------------------------------------------------------------------
# 3. Losses at training sizes: per-element bar against float64
# ---------------------------------------------------------------------------------------------------------------------

E_LOSS, TEMP = 768, 0.01


def _loss_inputs(B, F, Neg, F_total, seed):
    """q with |q| ~ 0.01 and doc rows of norm 2^k (k in [-8, 8] per (p, f)): scores stay within a few tens, so no
    softmax probability leaves fp32's normal range.  The mixture logits stay small (W ~ 3): their spread is covered
    by the mixture tests above, and here it would only add the weights' own rounding to every gradient row."""
    gen = torch.Generator().manual_seed(seed)
    sc = 1.0 / math.sqrt(E_LOSS)
    q = torch.randn(B, E_LOSS, generator=gen) * sc * 0.01
    dp = X.spread_rows(torch.randn(B, F, E_LOSS, generator=gen) * sc, gen)
    dn = X.spread_rows(torch.randn(B, F, Neg, E_LOSS, generator=gen) * sc, gen)
    W = torch.randn(E_LOSS, F_total, generator=gen) * 3.0
    return q, dp, dn, W


def _leaves(ts, device, dtype):
    return [t.to(device=device, dtype=dtype).clone().requires_grad_(True) for t in ts]


def _flip_e(ts):
    """q [B,E], docs [..,E], W [E,F]: the same problem with the E axis reversed (a second fp32 summation order)."""
    return [t.flip(0) if i == len(ts) - 1 else t.flip(-1) for i, t in enumerate(ts)]


def _unflip_grads(g):
    """loss, dq, dd_pos, dd_neg, dW of an E-reversed run, back in the original E order."""
    return [g[0], g[1].flip(-1), g[2].flip(-1), g[3].flip(-1), g[4].flip(0)]


def _check_grads(cuda, cpu32, f64, names):
    """Per-element bar of ``exact_train.row_bar``; rows are E-vectors (dW [E,F] is compared as dW^T)."""
    for c, a, b, n in zip(cuda, cpu32, f64, names):
        a = list(a)
        if n == "dW":
            c, a, b = c.t(), [x.t() for x in a], b.t()
        bar = X.row_bar(a, b)
        err = (c.detach().double().cpu() - b.detach().double().cpu()).abs()
        bad = err > bar
        assert not bad.any(), (f"{n}: {int(bad.sum())} of {bad.numel()} elements outside the bar, worst excess "
                               f"{float((err - bar).max()):.3g} (row max {float(b.abs().max()):.3g})")


LOSS_PAIRS = [(24, 8), (40, 22), (64, 44)]
DECOMPOSED_MODES = [("inbatch_reverse", True, True, 2), ("inbatch", True, False, 2), ("simple_neg1", False, True, 1),
                    ("simple_neg3", False, True, 3)]


@pytest.mark.parametrize("pair", [0, 1], ids=["a", "b"])
@pytest.mark.parametrize("mode", DECOMPOSED_MODES, ids=lambda m: m[0])
def test_decomposed_loss_per_element(mode, pair):
    L, _ = _mods()
    name, in_batch, reverse, Neg = mode
    B, F = LOSS_PAIRS[(DECOMPOSED_MODES.index(mode) + pair) % 3]
    q0, dp0, dn0, W0 = _loss_inputs(B, F, Neg, F, seed=B + F + Neg)
    outs = {}
    for key, dev, dt, flip in (("f64", DEV, torch.float64, False), ("cpu32", "cpu", torch.float32, False),
                               ("cpu32_rev", "cpu", torch.float32, True)):
        ins = [q0, dp0, dn0, W0]
        q, dp, dn, W = _leaves(_flip_e(ins) if flip else ins, dev, dt)
        loss = T.decomposed_loss(q, dp, dn, W, TEMP, True, reverse=reverse, in_batch_negative=in_batch)
        loss.backward()
        g = [loss.detach(), q.grad, dp.grad, dn.grad, W.grad]
        outs[key] = _unflip_grads(g) if flip else g
    q, dp, dn = _leaves((q0, dp0, dn0), DEV, torch.float32)
    layer = make_layer(W0, True)
    mod = L.DecomposedContrastiveLoss(temperature=TEMP, in_batch_negative=in_batch, reverse=reverse,
                                      all_gather_multi_gpu=False, mixture_of_fields_layer=layer)
    loss = mod(q, dp, dn)
    loss.backward()
    _check_grads([loss, q.grad, dp.grad, dn.grad, layer.weight.grad], zip(outs["cpu32"], outs["cpu32_rev"]),
                 outs["f64"], ["loss", "dq", "dd_pos", "dd_neg", "dW"])


def _hybrid_oracle(q, dp, dn, sp, W, bn):
    """HybridContrastiveLoss.forward (in-batch, reverse) on given sparse columns sp = (pos, neg, reverse-pos)."""
    B = q.shape[0]
    pos, neg = T.hybrid_scores(q, dp, dn, sp[0], sp[1], W, TEMP, True, bn)
    nll = T.sliced_nll(torch.cat([pos, neg], dim=1), B)
    rev_c = torch.cat([torch.einsum("pfe,be->bpf", dp, q) / TEMP, sp[2]], dim=-1)
    if bn is not None:
        rev_c = bn(rev_c.permute(0, 2, 1)).permute(0, 2, 1)
    return nll + T.sliced_nll(T.mixture(rev_c, q, W, True).t(), B)


def _sparse_indices(P, Neg, B, seed):
    """Two BM25sSparseIndex fields over the P + P*Neg docs, their doc keys and B query strings."""
    from mfar_b200.data.index import BM25sSparseIndex
    rng = np.random.RandomState(seed)
    words = [f"w{i}" for i in range(120)]
    keys = [f"d{i}" for i in range(P + P * Neg)]
    idx = {}
    for name, lo, hi in (("title", 2, 6), ("body", 8, 30)):
        docs = {k: " ".join(rng.choice(words, size=rng.randint(lo, hi))) for k in keys}
        idx[name] = BM25sSparseIndex.create(docs, device=DEV)
    queries = [" ".join(rng.choice(words, size=5)) for _ in range(B)]
    return idx, keys[:P], keys[P:], queries


HYBRID_MODES = [("nobn", False, None), ("bn", True, None), ("sparse_score_batch", True, "batch"),
                ("sparse_cache", True, "cache")]


@pytest.mark.parametrize("mode", HYBRID_MODES, ids=lambda m: m[0])
def test_hybrid_loss_per_element(mode):
    L, _ = _mods()
    name, use_bn, sparse = mode
    B, Fd = LOSS_PAIRS[HYBRID_MODES.index(mode) % 3]
    Neg = 2
    Fs = 2 if sparse else 0
    q0, dp0, dn0, W0 = _loss_inputs(B, Fd, Neg, Fd + Fs, seed=100 + B + Fd)
    query_ids = list(range(1000, 1000 + B))
    if sparse:
        idx, pos_keys, neg_keys, queries = _sparse_indices(B, Neg, B, seed=B)
        if sparse == "batch":
            sparse_scores = {"title": {7: {0: 1.0}}, "body": {}}          # the batch's query ids are missing
        else:
            sparse_scores = {}
            for fname, si in idx.items():
                per_q = {}
                for qid, text in zip(query_ids, queries):
                    s = si.get_scores(text)
                    per_q[qid] = {int(i): float(s[i]) for i in np.nonzero(s)[0]}
                sparse_scores[fname] = per_q
        calls = {fname: [] for fname in idx}
        for fname, si in idx.items():
            for meth in ("score_batch", "score_batch_with_cache"):
                orig = getattr(si, meth)

                def rec(*a, _orig=orig, _f=fname, **k):
                    r = _orig(*a, **k)
                    calls[_f].append(r)
                    return r
                setattr(si, meth, rec)
    else:
        idx, pos_keys, neg_keys, queries, sparse_scores = {}, ["d"] * B, ["n"] * (B * Neg), ["q"] * B, {}
    layer = make_layer(W0, True)
    mod = L.HybridContrastiveLoss(temperature=TEMP, all_gather_multi_gpu=False, mixture_of_fields_layer=layer,
                                  sparse_indices_dict=idx, num_fields=Fd + Fs, use_batchnorm=use_bn).to(DEV)
    bn0 = copy.deepcopy(mod.bn) if use_bn else None
    q, dp, dn = _leaves((q0, dp0, dn0), DEV, torch.float32)
    loss = mod(q, queries, dp, pos_keys, dn, neg_keys, query_ids, sparse_scores)
    loss.backward()
    if sparse:
        for fname in idx:
            assert len(calls[fname]) == 3, fname                         # pos, neg, reverse
            for c in calls[fname]:
                assert c.shape[0] == B and (c != 0).any()
        sp = [torch.stack([calls[f][i].double() for f in idx], dim=-1) for i in range(3)]
        assert sp[1].shape[1] == B * Neg
    else:
        sp = [torch.zeros(B, B, 0, dtype=torch.float64), torch.zeros(B, B * Neg, 0, dtype=torch.float64),
              torch.zeros(B, B, 0, dtype=torch.float64)]
    outs, bns = {}, {}
    for key, dev, dt, flip in (("f64", DEV, torch.float64, False), ("cpu32", "cpu", torch.float32, False),
                               ("cpu32_rev", "cpu", torch.float32, True)):
        ins = [q0, dp0, dn0, W0]
        qq, dpp, dnn, WW = _leaves(_flip_e(ins) if flip else ins, dev, dt)
        bn = copy.deepcopy(bn0).to(device=dev, dtype=dt) if use_bn else None
        l_ = _hybrid_oracle(qq, dpp, dnn, [s.to(device=dev, dtype=dt) for s in sp], WW, bn)
        l_.backward()
        g = [l_.detach(), qq.grad, dpp.grad, dnn.grad, WW.grad]
        outs[key] = _unflip_grads(g) if flip else g
        bns[key] = bn
    _check_grads([loss, q.grad, dp.grad, dn.grad, layer.weight.grad], zip(outs["cpu32"], outs["cpu32_rev"]),
                 outs["f64"], ["loss", "dq", "dd_pos", "dd_neg", "dW"])
    if use_bn:
        _check_grads([mod.bn.running_mean, mod.bn.running_var],
                     [(bns[k].running_mean for k in ("cpu32", "cpu32_rev")),
                      (bns[k].running_var for k in ("cpu32", "cpu32_rev"))],
                     [bns["f64"].running_mean, bns["f64"].running_var], ["running_mean", "running_var"])
        assert int(mod.bn.num_batches_tracked) == 2
