#!/usr/bin/env python
"""Randomised parity sweep of the scoring kernels against the CPU oracle (needs a B200; not part of pytest).

    python tools/fuzz_parity.py --seconds 120 --seed 0 --out gpurun_out/fuzz.json

Draws shapes across the envelope every kernel claims (doc counts around the 128-doc tile and 64-doc half-tile
boundaries, dims 32..1024 incl. ones that are not a multiple of 64, 0..6 dense and 0..3 sparse fields, batches around
the 16/32/64/128/256 query-tile boundaries, k 1..128, masks, doc-id bases, f16/f32 sparse inputs, all four impl
requests) and applies the same assertion as tests/parity.py.  Every failure is recorded with its parameters; the
exit code is the number of failures (0 = clean).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (os.path.join(ROOT, "multifield-adaptive-retrieval_b200"), os.path.join(ROOT, "oracle"),
           os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import mfar_oracle as O  # noqa: E402  (checker)
from parity import assert_same_topk_up_to_ties, assert_topk_parity  # noqa: E402


def _term_scale(c: dict) -> float:
    """Typical magnitude of ONE weighted per-field term of the mixture score (dense dot of N(0,1)-ish vectors ~ sqrt(d),
    weight ~ 1/F): the floor of the scale tolerances are taken relative to, so that a tiny shard whose scores happen to
    be near-zero cancellations of such terms is judged against the terms, not against the cancellation."""
    if c.get("normalize") or c["Fd"] == 0:
        return 0.0
    return 0.05 * float(np.sqrt(c["d"])) / (c["Fd"] + c["Fs"])


def draw_case(rng: np.random.RandomState) -> dict:
    n_choices = [1, 2, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 256, 257, 1000, 4095, 4097]
    N = int(rng.choice(n_choices)) if rng.rand() < 0.6 else int(rng.randint(1, 20000))
    d = int(rng.choice([32, 64, 100, 128, 192, 256, 320, 768, 1024]))
    Fd = int(rng.choice([0, 1, 1, 2, 3, 5, 6]))
    Fs = int(rng.choice([0, 0, 1, 2, 3]))
    if Fd + Fs == 0:
        Fd = 1
    q_choices = [1, 2, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 300]
    Q = int(rng.choice(q_choices))
    if N * max(Fd, 1) * d > 2.5e7 or Q * N * max(Fs, 1) > 1.2e7:       # keep the fp32 oracle in the seconds range
        N = max(1, min(N, int(2.5e7 / (max(Fd, 1) * d)), int(1.2e7 / (Q * max(Fs, 1)))))
    k = int(min(N, rng.choice([1, 2, 10, 50, 100, 100, 127, 128])))
    impl = str(rng.choice(["auto", "simt", "tcgen05", "tcgen05_qs"]))
    if Fd == 0 or d % 64 != 0:                                          # tensor-core paths need dim % 64 == 0 ...
        impl = str(rng.choice(["auto", "simt"]))                        # (PackedCorpus pads dim, so "auto" still may)
    if impl == "tcgen05_qs" and d > 768:                                # queries must fit 384 TMEM columns
        impl = "tcgen05"
    return dict(N=N, d=d, Fd=Fd, Fs=Fs, Q=Q, k=k, impl=impl, query_cond=bool(rng.rand() < 0.6),
                base=int(rng.choice([0, 0, 12345, 3_000_000_000])), sparse_f32=bool(rng.rand() < 0.4),
                n_masked=int(rng.randint(0, 2)) if Fd + Fs > 1 else 0, normalize=bool(rng.rand() < 0.15),
                seed=int(rng.randint(0, 2 ** 31 - 1)))


def run_case(c: dict) -> None:
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    dev = "cuda"
    g = torch.Generator().manual_seed(c["seed"])
    N, d, Fd, Fs, Q, k = c["N"], c["d"], c["Fd"], c["Fs"], c["Q"], c["k"]
    mu = torch.randn(d, generator=g)
    raw = [torch.randn(N, d, generator=g) + 0.5 * mu for _ in range(Fd)]
    qraw = torch.randn(Q, d, generator=g) + 0.5 * mu
    if c["normalize"]:                              # oracle side of Normalize(): float64 normalise, one bf16 rounding
        fields = [torch.from_numpy(O.normalize_rows_bf16(f)) for f in raw]
        q = torch.from_numpy(O.normalize_rows_bf16(qraw))
    else:
        fields = [O.round_bf16(f) for f in raw]
        q = O.round_bf16(qraw)
        raw, qraw = fields, q
    sp = None
    if Fs:
        u = torch.rand(Q, Fs, N, generator=g)
        sp = torch.where(u < 0.9, torch.zeros(()), 8.0 * torch.rand(Q, Fs, N, generator=g)).half()
    F = Fd + Fs
    qc = c["query_cond"]
    W = 0.05 * torch.randn(d, F, generator=g) if qc else torch.randn(F, 1, generator=g)
    layer = LinearWeights(d, F, query_cond=True) if qc else LinearWeights(F, 1)
    with torch.no_grad():
        layer.weight.copy_(W)
    pc = PackedCorpus.from_fields(raw, dev, c["normalize"]) if Fd else None
    r = MultiFieldRetriever(pc, layer.to(dev), n_sparse=Fs, top_k=k, doc_id_base=c["base"], impl=c["impl"], n_docs=N,
                            device=dev)
    mask = torch.ones(F, 1)
    if c["n_masked"]:
        idx = [int(c["seed"] % F)]
        mask[idx] = 0
        r.mask_field(idx)
    sp_in = None if sp is None else (sp.float() if c["sparse_f32"] else sp).to(dev)
    q_emb = qraw.to(dev) if not c["normalize"] else q.to(dev)
    scores, ids = r.search(qraw.to(dev) if Fd else None, q_emb, sp_in)
    torch.cuda.synchronize()
    w = O.mixture_weights(q_emb.float().cpu() if qc else None, W, qc)
    ref = O.exhaustive_scores(q, fields, None if sp is None else sp.float(), w, mask)
    assert_topk_parity(scores.cpu().numpy(), ids.cpu().numpy(), ref.numpy(), k, id_offset=c["base"], rtol=2e-5,
                       tie_rel=1e-5, scale_floor=_term_scale(c))


def draw_api_case(rng: np.random.RandomState) -> dict:
    c = draw_case(rng)
    c["impl"] = "auto"
    c["normalize"] = False
    c["Fd"] = max(1, c["Fd"])
    c["N"] = max(c["N"], 2)
    c["k"] = int(min(c["k"], c["N"]))
    c["base"] = int(rng.choice([0, 777]))
    return c


def run_api_case(c: dict) -> None:
    """One shape through every entry path that must agree: device search, the host-buffer C call, the COO sparse
    input, doc-range shards + merge, the CUDA-graph replay, the one-pass mask sweep, per-field top-k, union_rescore."""
    from mfar_b200.dist import merge_keys
    from mfar_b200.modeling.retrieval import GraphedSearch, MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    dev = "cuda"
    g = torch.Generator().manual_seed(c["seed"])
    N, d, Fd, Fs, Q, k, base = c["N"], c["d"], c["Fd"], c["Fs"], c["Q"], c["k"], c["base"]
    mu = torch.randn(d, generator=g)
    fields = [O.round_bf16(torch.randn(N, d, generator=g) + 0.5 * mu) for _ in range(Fd)]
    q = O.round_bf16(torch.randn(Q, d, generator=g) + 0.5 * mu)
    sp = None
    if Fs:
        u = torch.rand(Q, Fs, N, generator=g)
        sp = torch.where(u < 0.9, torch.zeros(()), 8.0 * torch.rand(Q, Fs, N, generator=g)).half()
    F = Fd + Fs
    qc = c["query_cond"]
    W = 0.05 * torch.randn(d, F, generator=g) if qc else torch.randn(F, 1, generator=g)
    layer = LinearWeights(d, F, query_cond=True) if qc else LinearWeights(F, 1)
    with torch.no_grad():
        layer.weight.copy_(W)
    layer = layer.to(dev)

    def make(lo, hi):
        return MultiFieldRetriever(PackedCorpus.from_fields([f[lo:hi] for f in fields], dev), layer, n_sparse=Fs,
                                   top_k=k, doc_id_base=base + lo)
    r = make(0, N)
    mask = torch.ones(F, 1)
    if c["n_masked"]:
        idx = [int(c["seed"] % F)]
        mask[idx] = 0
        r.mask_field(idx)
    qd, spd = q.to(dev), (None if sp is None else sp.to(dev))
    w = O.mixture_weights(q if qc else None, W, qc)
    ref = O.exhaustive_scores(q, fields, None if sp is None else sp.float(), w, mask).numpy()
    s0, i0, k0 = r.search(qd, qd, spd, return_keys=True)
    assert_topk_parity(s0.cpu().numpy(), i0.cpu().numpy(), ref, k, id_offset=base, scale_floor=_term_scale(c))
    # host-buffer C call == device call, bit for bit
    qh = r.corpus.prepare_queries(q).cpu().pin_memory()
    s_h, i_h = r.search_host(qh, q.float().pin_memory() if qc else None, None if sp is None else sp.pin_memory())

    def same(sa, ia, sb, ib, what):
        """Entry paths that run the same kernels agree bit for bit.  With sparse fields the paths may differ in WHERE the
        sparse term is added (row pitch 32-byte aligned: gathered inside the scoring epilogue, and the query-stationary
        epilogue interleaves it with the dense fields; otherwise pre-mixed first), i.e. in fp32 summation order."""
        if Fs and Fd:
            assert_same_topk_up_to_ties(sa.cpu(), ia.cpu(), sb.cpu(), ib.cpu())
        else:
            assert torch.equal(sa.cpu(), sb.cpu()) and torch.equal(ia.cpu(), ib.cpu()), what
    same(s_h, i_h, s0, i0, "search_host != search")
    # COO sparse input (global doc ids) vs the oracle
    if Fs:
        ks, vs, offs = [], [], [0]
        for j in range(Fs):
            nz = torch.nonzero(sp[:, j, :])
            ks.append(torch.stack([nz[:, 0], nz[:, 1] + base], dim=1).int())
            vs.append(sp[nz[:, 0], j, nz[:, 1]])
            offs.append(offs[-1] + len(nz))
        coo = (torch.cat(ks).to(dev), torch.cat(vs).to(dev), offs)
        s_c, i_c = r.search(qd, qd, sparse_coo=coo)
        assert_topk_parity(s_c.cpu().numpy(), i_c.cpu().numpy(), ref, k, id_offset=base, scale_floor=_term_scale(c))
    # doc-range shards (arbitrary, not tile-aligned cut) merged == unsharded, bit for bit
    cut = 1 + int(c["seed"] % (N - 1))
    keys = []
    for lo, hi in ((0, cut), (cut, N)):
        sh = make(lo, hi)
        sh.mask = r.mask
        kk = sh.search(qd, qd, None if spd is None else spd[:, :, lo:hi].contiguous(), top_k=min(k, hi - lo),
                       return_keys=True)[2]
        keys.append(torch.nn.functional.pad(kk, (0, k - kk.shape[1])))
    s_m, i_m = merge_keys(torch.stack(keys), k)
    same(s_m, i_m, s0, i0, "shard merge != unsharded")
    # CUDA-graph replay == eager
    gs = GraphedSearch(r, Q, sparse="dense" if Fs else "none", sparse_ld=None if sp is None else N)
    s_g, i_g = gs(qd, qd.float(), sparse=spd)
    same(s_g, i_g, s0, i0, "graph replay != eager")
    # one-pass mask sweep == mask_field loop (vs the oracle)
    if F > 1:
        sets = [[], [0], [F - 1], list(range(0, F, 2))]
        S, I = r.search_mask_sweep(qd, sets, qd, spd, max_rows=max(Q, 300))
        for m, idx in enumerate(sets):
            mm = torch.ones(F, 1)
            mm[idx] = 0
            ref_m = O.exhaustive_scores(q, fields, None if sp is None else sp.float(), w, mm).numpy()
            assert_topk_parity(S[m].cpu().numpy(), I[m].cpu().numpy(), ref_m, k, id_offset=base,
                               scale_floor=_term_scale(c))
    # per-field top-k incl. the zero-init quirk, and the faithful union_rescore pipeline, vs the oracle
    ps, pr = r.per_field_topk(qd, spd, k)
    for f in range(Fd):
        rs, rr = O.dense_retrieve_batch(q, fields[f], k)
        np.testing.assert_allclose(ps[f].cpu().numpy(), rs.numpy(), rtol=2e-5, atol=2e-5 * float(rs.abs().max() + 1e-30))
    if Q <= 33 and Fs == 0:                 # (sparse per-field top-k reaches into exact-zero ties: union order unpinned)
        try:
            want_v, want_r = O.union_rescore(q, fields, None if sp is None else sp.float(), q if qc else None, W, qc,
                                             mask, k)
        except RuntimeError:
            want_v = None                       # union smaller than k: the reference's torch.topk raises
        if want_v is not None:
            got_v, got_r = r.union_rescore(qd, qd, spd)
            for i in range(Q):
                wv = want_v[i].numpy()
                np.testing.assert_allclose(got_v[i].cpu().numpy(), wv, rtol=2e-5, atol=2e-5 * float(np.abs(wv).max() + 1e-30))
    torch.cuda.synchronize()


def draw_bm25_case(rng: np.random.RandomState) -> dict:
    return dict(N=int(rng.choice([1, 2, 127, 128, 129, 1000, 4096, 4097, int(rng.randint(3, 12000))])),
                V=int(rng.choice([1, 2, 7, 50, 300, 3000])), mean_len=int(rng.choice([1, 3, 10, 40])),
                Fs=int(rng.choice([1, 2, 3])), Fd=int(rng.choice([0, 1, 2])), d=int(rng.choice([64, 128])),
                Q=int(rng.choice([1, 3, 17, 64, 65, 130])), n_tok=int(rng.choice([1, 3, 8, 20])),
                k=int(rng.choice([1, 10, 100, 128])), shard=bool(rng.rand() < 0.5), impl="auto",
                seed=int(rng.randint(0, 2 ** 31 - 1)))


def run_bm25_case(c: dict) -> None:
    """Device BM25 (index build, get_scores, hybrid search from query tokens, doc-range shard, pair producer) vs the
    numpy BM25 oracle."""
    import bm25_oracle as B
    import precompute_oracle as PO
    from mfar_b200.data.bm25 import DeviceBM25, rows_to_coo, safe_docs_bitmap
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    dev = "cuda"
    rng = np.random.default_rng(c["seed"])
    N, V, Fs, Fd, d, Q = c["N"], c["V"], c["Fs"], c["Fd"], c["d"], c["Q"]
    k = min(c["k"], N)
    p = 1.0 / np.arange(1, V + 1)
    p /= p.sum()
    corpora = [[rng.choice(V, size=max(1, rng.poisson(c["mean_len"])), p=p).tolist() for _ in range(N)] for _ in range(Fs)]
    tokens = [[rng.choice(V + 3, size=rng.integers(0, c["n_tok"] + 1)).tolist() for _ in range(Q)] for _ in range(Fs)]
    bm = [DeviceBM25(device=dev).index(cp, vocab=V) for cp in corpora]
    oidx = [B.build_index(cp, V) for cp in corpora]
    for j in range(Fs):                                           # index: structure bit-exact, values within 1 ulp
        sc = bm[j].scores
        assert np.array_equal(sc["indptr"].cpu().numpy(), oidx[j]["indptr"]), "indptr"
        assert np.array_equal(sc["indices"].cpu().numpy(), oidx[j]["indices"]), "indices"
        np.testing.assert_allclose(sc["data"].cpu().numpy(), oidx[j]["data"], rtol=2.4e-7, atol=0)
    want = np.stack([[B.get_scores(oidx[j], [t for t in tokens[j][q] if t < V]) for j in range(Fs)] for q in range(Q)])
    got = bm[0].get_scores_batch(tokens[0]).cpu().numpy()
    np.testing.assert_allclose(got, want[:, 0], rtol=4e-6, atol=1e-6)
    assert np.array_equal(got == 0, want[:, 0] == 0), "zero pattern"
    # pair producer on the device rows vs the CPU restatement on the SAME rows (bit-exact)
    safe = set(rng.choice(N, size=max(1, N // 2), replace=False).tolist())
    rows_dev = bm[0].get_scores_batch(tokens[0])
    kk, vv = rows_to_coo(rows_dev, N, torch.from_numpy(safe_docs_bitmap(safe, N).view(np.int32)).to(dev),
                         torch.arange(Q, dtype=torch.int32) * 7, 0)
    rows_host = rows_dev.cpu().numpy()
    wk, wv = PO.precompute_score_for_field({7 * q: rows_host[q] for q in range(Q)}, safe)
    assert np.array_equal(kk.cpu().numpy(), wk) and np.array_equal(vv.cpu().numpy().view(np.uint16), wv.view(np.uint16)), "coo"
    # hybrid search from tokens vs the oracle
    g = torch.Generator().manual_seed(c["seed"])
    fields = [O.round_bf16(torch.randn(N, d, generator=g)) for _ in range(Fd)]
    q = O.round_bf16(torch.randn(Q, d, generator=g))
    F = Fd + Fs
    W = 0.05 * torch.randn(d, F, generator=g)
    layer = LinearWeights(d, F, query_cond=True)
    with torch.no_grad():
        layer.weight.copy_(W)
    layer = layer.to(dev)
    w = O.mixture_weights(q, W, True)
    ref = O.exhaustive_scores(q, fields, torch.from_numpy(want), w).numpy()
    lo, hi = (0, N)
    if c["shard"] and N >= 4:
        lo, hi = N // 4, N - N // 3
    k = min(k, hi - lo)
    pc = PackedCorpus.from_fields([f[lo:hi] for f in fields], dev) if Fd else None
    r = MultiFieldRetriever(pc, layer, top_k=k, doc_id_base=lo, n_docs=hi - lo, device=dev,
                            sparse_indices=[b.shard(lo, hi) for b in bm] if (lo, hi) != (0, N) else bm)
    s, i = r.search(q.to(dev) if Fd else None, q.to(dev), sparse_tokens=tokens)
    assert_topk_parity(s.cpu().numpy(), i.cpu().numpy(), ref[:, lo:hi], k, id_offset=lo, rtol=2e-5,
                       scale_floor=_term_scale(c))
    torch.cuda.synchronize()


def draw_train_case(rng: np.random.RandomState) -> dict:
    Neg = int(rng.choice([1, 1, 2, 4]))
    F = int(rng.choice([1, 2, 5, 22])) if Neg == 1 else int(rng.choice([1, 1, 3]))
    return dict(B=int(rng.choice([1, 2, 12, 31, 32, 33, 64, 100])), P=int(rng.choice([1, 2, 12, 33, 70])), F=F, Neg=Neg,
                E=int(rng.choice([4, 64, 100, 256, 768, 1024])), query_cond=bool(rng.rand() < 0.5), impl="train",
                seed=int(rng.randint(0, 2 ** 31 - 1)))


def run_train_case(c: dict) -> None:
    """Training-time scorer forward + backward (csrc/train.cu) vs the torch CPU oracle with autograd."""
    import train_oracle as T
    from mfar_b200.modeling import losses as L
    from mfar_b200.modeling.weighting import LinearWeights
    dev = "cuda"
    B_, P, F, Neg, E, qc = c["B"], c["P"], c["F"], c["Neg"], c["E"], c["query_cond"]
    g = torch.Generator().manual_seed(c["seed"])
    sc = 1.0 / np.sqrt(E)
    q0, dp0 = torch.randn(B_, E, generator=g) * sc, torch.randn(P, F, E, generator=g) * sc
    dn0 = torch.randn(P, F, Neg, E, generator=g) * sc
    W0 = torch.randn(E, F, generator=g) * 0.5 if qc else torch.randn(F, 1, generator=g)
    temp = 0.05
    q, dp, dn, W = (t.clone().requires_grad_(True) for t in (q0, dp0, dn0, W0))
    if Neg > 1 and F > 1:
        return                                     # the reference's .view raises for this layout (losses.py:186)
    pc, nc = T.field_components(q, dp, dn, temp)
    scores = torch.cat([T.mixture(pc, q, W, qc), T.mixture(nc, q, W, qc)], dim=1)
    go = torch.randn(scores.shape, generator=g)
    (scores * go).sum().backward()
    cq, cdp, cdn = (t.clone().to(dev).requires_grad_(True) for t in (q0, dp0, dn0))
    layer = LinearWeights(W0.shape[0], W0.shape[1], query_cond=qc)
    with torch.no_grad():
        layer.weight.copy_(W0)
    layer = layer.to(dev)
    mod = L.DecomposedContrastiveLoss(temperature=temp, all_gather_multi_gpu=False, mixture_of_fields_layer=layer)
    sp, sn = mod.compute_query_doc_scores(cq, cdp, cdn)
    cs = torch.cat([sp, sn], dim=1)

    def close(a, b, what, rtol, floor):
        # scale floor: a one-doc / one-query batch can make a whole tensor a near-zero cancellation of O(floor) terms
        a, b = a.detach().cpu().double().numpy(), b.detach().double().numpy()
        assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
        scale = max(np.abs(b).max(), floor, 1e-30)
        assert np.abs(a - b).max() <= rtol * scale, f"{what}: max abs diff {np.abs(a - b).max()} vs scale {scale}"
    comp_scale = float(max(pc.detach().abs().max(), nc.detach().abs().max()))
    close(cs, scores, "scores", 1e-5, 0.05 * comp_scale)
    (cs * go.to(dev)).sum().backward()
    grad_scale = 0.02 * float(max(t.grad.abs().max() for t in (q, dp, dn, W)))
    close(cq.grad, q.grad, "dq", 1e-4, grad_scale)
    close(cdp.grad, dp.grad, "dd_pos", 1e-4, grad_scale)
    close(cdn.grad, dn.grad, "dd_neg", 1e-4, grad_scale)
    close(layer.weight.grad, W.grad, "dW", 1e-4, grad_scale)
    torch.cuda.synchronize()


MODES = {"kernels": (draw_case, run_case), "api": (draw_api_case, run_api_case),
         "bm25": (draw_bm25_case, run_bm25_case), "train": (draw_train_case, run_train_case)}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="kernels", choices=sorted(MODES))
    ap.add_argument("--seconds", type=float, default=120.0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "fuzz.json"))
    args = ap.parse_args()
    rng = np.random.RandomState(args.seed)
    t0 = time.time()
    n, failures, per_impl = 0, [], {}
    while time.time() - t0 < args.seconds:
        c = MODES[args.mode][0](rng)
        n += 1
        per_impl[c["impl"]] = per_impl.get(c["impl"], 0) + 1
        try:
            MODES[args.mode][1](c)
        except Exception as e:  # noqa: BLE001  (recorded, sweep goes on)
            failures.append(dict(case=c, error=f"{type(e).__name__}: {e}"[:600], trace=traceback.format_exc()[-1500:]))
            print("FAIL", json.dumps(c), str(e)[:200], flush=True)
            if "CUDA error" in str(e) or "illegal" in str(e).lower():
                break                                                   # sticky context error: nothing more to learn
    res = dict(mode=args.mode, cases=n, failures=len(failures), seconds=round(time.time() - t0, 1), per_impl=per_impl, seed=args.seed,
               failed=failures)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "failed"}))
    return len(failures)


if __name__ == "__main__":
    sys.exit(min(main(), 100))
