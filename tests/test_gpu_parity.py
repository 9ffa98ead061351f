"""CUDA path vs oracle / reference-generated golden vectors.  Every call goes through the C ABI
(ctypes -> libmfar_b200.so).  Bar: ids identical except near-ties, scores within 1e-2 relative of
the fp32 reference on identical bf16-rounded inputs (asserted at 2e-5, tests/parity.py)."""
import glob
import io
import json
import os

import numpy as np
import pytest
import torch

import mfar_oracle as O
from parity import assert_same_topk_up_to_ties, assert_topk_parity

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = sorted(glob.glob(os.path.join(GOLDEN, "*.npz")))
IMPLS = ["simt", "tcgen05", "tcgen05_qs"]
DEV = "cuda"


def _mods():
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    return MultiFieldRetriever, PackedCorpus, LinearWeights


def load(path):
    z = np.load(path, allow_pickle=False)
    return z, json.loads(str(z["meta"]))


def build(fields, W, query_cond, n_sparse=0, k=100, normalize=False, doc_id_base=0, impl="auto", n_docs=None):
    MultiFieldRetriever, PackedCorpus, LinearWeights = _mods()
    pc = PackedCorpus.from_fields(fields, DEV, normalize) if len(fields) else None
    F = len(fields) + n_sparse
    layer = LinearWeights(W.shape[0], W.shape[1], query_cond=True) if query_cond else LinearWeights(F, 1)
    with torch.no_grad():
        layer.weight.copy_(torch.as_tensor(W))
    layer = layer.to(DEV)
    n_docs = fields[0].shape[0] if len(fields) else n_docs
    return MultiFieldRetriever(pc, layer, n_sparse=n_sparse, top_k=k, doc_id_base=doc_id_base, impl=impl,
                               n_docs=n_docs, device=DEV)


def synth(seed, N, d, Fd, Fs, Q, query_cond=True):
    g = torch.Generator().manual_seed(seed)
    mu = torch.randn(d, generator=g)
    fields = [O.round_bf16(torch.randn(N, d, generator=g) + 0.5 * mu) for _ in range(Fd)]
    q = O.round_bf16(torch.randn(Q, d, generator=g) + 0.5 * mu)
    sp = None
    if Fs:
        u = torch.rand(Q, Fs, N, generator=g)
        gam = -2.0 * (torch.log(torch.rand(Q, Fs, N, generator=g)) + torch.log(torch.rand(Q, Fs, N, generator=g)))
        sp = torch.where(u < 0.95, torch.zeros(()), gam).half()
    F = Fd + Fs
    W = 0.05 * torch.randn(d, F, generator=g) if query_cond else torch.randn(F, 1, generator=g)
    return fields, q, sp, W


# ----------------------------------------------------------------------------------------------
def test_device_is_sm100_and_library_loaded():
    from mfar_b200 import _native as nv
    assert nv.lib().mfar_device_check(-1) == 0
    assert torch.cuda.get_device_capability()[0] == 10


def test_pack_unpack_roundtrip_bit_exact():
    _, PackedCorpus, _ = _mods()
    g = torch.Generator().manual_seed(1)
    for N, d, F in [(300, 64, 3), (129, 768, 2), (128, 32, 1)]:
        fields = [torch.randn(N, d, generator=g) for _ in range(F)]
        pc = PackedCorpus.from_fields(fields, DEV)
        for f in range(F):
            got = pc.unpack_field(f).cpu()
            assert torch.equal(got, fields[f].to(torch.bfloat16).float())
        assert pc.data.numel() == ((N + 127) // 128) * F * 128 * pc.dim_pad


@pytest.mark.parametrize("query_cond", [True, False])
def test_mixture_weights_and_forward_match_oracle(query_cond):
    _, _, LinearWeights = _mods()
    g = torch.Generator().manual_seed(2)
    B, S, E, F = 5, 37, 768, 22
    W = 0.05 * torch.randn(E, F, generator=g) if query_cond else torch.randn(F, 1, generator=g)
    q = torch.randn(B, E, generator=g)
    x = torch.randn(B, S, F, generator=g)
    layer = LinearWeights(E, F, query_cond=True) if query_cond else LinearWeights(F, 1)
    with torch.no_grad():
        layer.weight.copy_(W)
    layer = layer.to(DEV)
    mask = torch.ones(F, 1)
    mask[3] = 0
    w = layer.field_weights(q.to(DEV) if query_cond else None, mask.to(DEV), batch=B).cpu()
    ref_w = O.mixture_weights(q, W, query_cond).expand(B, F) * mask.reshape(1, F)
    torch.testing.assert_close(w, ref_w, rtol=2e-5, atol=1e-7)
    out = layer(x.to(DEV), q.to(DEV) if query_cond else None).cpu()
    torch.testing.assert_close(out, O.linear_weights_forward(x, q, W, query_cond), rtol=2e-5, atol=1e-5)
    out2 = layer(x[0].to(DEV), q[:1].to(DEV) if query_cond else None).cpu()          # [S,F] form of trec_eval_step
    assert out2.shape == (1, S)
    torch.testing.assert_close(out2, O.linear_weights_forward(x[0], q[:1], W, query_cond), rtol=2e-5, atol=1e-5)


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_exhaustive_search_vs_reference_golden(path, impl):
    """Top-k of the CUDA path against the all-doc mixture scores the REFERENCE's own LinearWeights /
    DenseFlatIndex / BM25sSparseIndex.score_batch produced (tests/golden, ref_mix_all)."""
    z, m = load(path)
    fields = [torch.from_numpy(z["fields"][f]) for f in range(m["Fd"])]
    sp = torch.from_numpy(z["sparse"]).to(DEV) if m["Fs"] else None
    k = m["k"]
    r = build(fields, z["W"], m["query_cond"], m["Fs"], k, impl=impl)
    r.mask = torch.from_numpy(z["mask"]).to(DEV)
    q = torch.from_numpy(z["q"])
    scores, ids = r.search(q.to(DEV), q.to(DEV), sp)
    assert_topk_parity(scores.cpu().numpy(), ids.cpu().numpy(), z["ref_mix_all"], k)
    # fp16 and fp32 sparse inputs agree (golden sparse values are fp16-representable)
    if sp is not None:
        s2, i2 = r.search(q.to(DEV), q.to(DEV), sp.half())
        assert torch.equal(i2, ids) and torch.equal(s2, scores)


SHAPES = [
    # seed, N, d, Fd, Fs, Q, query_cond, k
    (21, 2000, 768, 22, 0, 64, True, 100),      # config 1 shape (PRIME truncated, all_dense, dev batch 64)
    (22, 1500, 768, 5, 0, 1, True, 100),        # MAG-shaped, batch 1
    (23, 1111, 768, 8, 8, 3, True, 100),        # Amazon-shaped hybrid, ragged N
    (24, 900, 768, 1, 0, 5, False, 100),        # single_dense, static weights
    (25, 700, 768, 0, 4, 6, False, 50),         # sparse only: streaming top-k of the pre-mixed rows (topk_rows.cu)
    (32, 70000, 64, 0, 3, 9, True, 100),        # sparse only, seeded thresholds, several segments per row, ragged tail
    (33, 4097, 64, 0, 1, 130, False, 128),      # sparse only, k = 128, just above the seeding size, N % 4 == 1
    (26, 3000, 768, 3, 2, 70, True, 100),       # Q > 64: two query tiles on the tcgen05 path
    (27, 129, 64, 2, 1, 17, True, 100),         # 2 tiles, the second with a single doc
    (28, 128, 128, 4, 0, 33, True, 128),        # k = 128 = N (everything returned)
    (29, 5000, 256, 2, 0, 130, True, 10),       # three query tiles
    (30, 4000, 768, 3, 1, 200, True, 100),      # large batch, hybrid: CTA-pair query-stationary path under auto
    (31, 2500, 768, 2, 0, 300, False, 100),     # 3 query tiles of 128 -> padded to 2 pairs
    (34, 6000, 768, 1, 0, 300, True, 100),      # single_ scorer, CTA pairs: two epilogue sets (score_qs_kernel<2,2>)
    (35, 3001, 256, 1, 2, 257, False, 100),     # single dense + 2 sparse fields, pairs + sparse base, ragged last tile
    (36, 700, 128, 1, 0, 129, True, 128),       # single field, k = 128, Q just above one query tile
]


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("shape", SHAPES, ids=[f"s{s[0]}" for s in SHAPES])
def test_exhaustive_search_vs_oracle(shape, impl):
    seed, N, d, Fd, Fs, Q, qc, k = shape
    if impl != "simt" and Fd == 0:
        pytest.skip("sparse-only batches have no dense contraction: every impl request runs topk_rows.cu")
    fields, q, sp, W = synth(seed, N, d, Fd, Fs, Q, qc)
    r = build(fields, W, qc, Fs, k, impl=impl, n_docs=N)
    mask = torch.ones(Fd + Fs, 1)
    if Fd + Fs > 2:
        mask[1] = 0
        r.mask_field([1])
    scores, ids = r.search(q.to(DEV) if Fd else None, q.to(DEV), None if sp is None else sp.to(DEV))
    w = O.mixture_weights(q if qc else None, W, qc)
    ref = O.exhaustive_scores(q, fields, None if sp is None else sp.float(), w, mask) if Fd else \
        O.exhaustive_scores(q, [], sp.float(), w, mask)
    assert_topk_parity(scores.cpu().numpy(), ids.cpu().numpy(), ref.numpy(), k)


def _ranked_case(N, F, d, Q, seed, k=100):
    """Corpus-sized synthetic shard + the fp32 checker's exact top-(k+slack) (tests/checker.py)."""
    MultiFieldRetriever, PackedCorpus, LinearWeights = _mods()
    from checker import Fp32Checker
    from mfar_b200 import synth as S
    pc = PackedCorpus(N, F, d, DEV)
    S.fill_packed_corpus(pc, seed=seed)
    mu = S.corpus_mean(d, seed, DEV)
    q = S.make_queries(Q, d, mu, seed + 1, DEV)
    layer = LinearWeights(d, F, query_cond=True)
    with torch.no_grad():
        layer.weight.copy_(S.make_mixture(d, F, seed + 2))
    r = MultiFieldRetriever(pc, layer.to(DEV), top_k=k)
    w = O.mixture_weights(q.float().cpu(), layer.weight.detach().cpu(), True).to(DEV)
    chk = Fp32Checker(pc)
    ref_s, ref_i = chk.topk(q, w, k, slack=64)
    return r, q, w, chk, ref_s, ref_i


def _assert_ranked(r, q, w, chk, ref_s, ref_i, impl, k=100):
    from checker import assert_topk_parity_at_scale
    n = q.shape[0]
    s, i = r.search(q, q.float(), impl=impl)
    assert_topk_parity_at_scale(s, i, ref_s[:n], ref_i[:n], chk.rescore(q, w[:n], i), k, r.n_docs, what=impl)
    return s, i


def test_simt_and_tcgen05_ranked_at_scale():
    """Both CUDA paths over 200k docs x 4 fields - a size the CPU oracle would take minutes for - ranked against the
    fp32 checker with the near-tie rule (a dropped winner fails), not merely compared with each other."""
    r, q, w, chk, ref_s, ref_i = _ranked_case(200_000, 4, 768, 4, 7)
    for impl in ("simt", "tcgen05"):
        _assert_ranked(r, q, w, chk, ref_s, ref_i, impl)


def test_query_stationary_and_doc_stationary_ranked_at_scale():
    """Large-batch kernel (queries in TMEM, CTA pairs) and the doc-stationary tcgen05 kernel over 150k docs x 3
    fields at Q=384, each ranked against the fp32 checker."""
    r, q, w, chk, ref_s, ref_i = _ranked_case(150_000, 3, 768, 384, 17)
    for impl in ("tcgen05", "tcgen05_qs"):
        _assert_ranked(r, q, w, chk, ref_s, ref_i, impl)


def test_single_field_two_epilogue_sets_ranked_at_scale():
    """single_ scorer at Q=384 (CTA pairs, two epilogue sets with their own candidate lists) ranked against the fp32
    checker; also Q=1024 against itself split into two batches (bit-identical)."""
    r, q, w, chk, ref_s, ref_i = _ranked_case(400_000, 1, 768, 1024, 27)
    for impl in ("tcgen05", "tcgen05_qs"):
        _assert_ranked(r, q[:384], w, chk, ref_s, ref_i, impl)
    sa, ia = _assert_ranked(r, q, w, chk, ref_s, ref_i, "auto")
    sb, ib = r.search(q[:512], q[:512].float())
    sc, ic = r.search(q[512:], q[512:].float())
    assert torch.equal(ia, torch.cat([ib, ic])) and torch.equal(sa, torch.cat([sb, sc]))


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_per_field_topk_vs_reference_retrieve_batch(path):
    """DenseFlatIndex.retrieve_batch incl. the (0.0, row 0) running-top-k init (index.py:192-193)."""
    z, m = load(path)
    if m["Fd"] == 0:
        pytest.skip("no dense field")
    fields = [torch.from_numpy(z["fields"][f]) for f in range(m["Fd"])]
    r = build(fields, np.ones((m["Fd"], 1), np.float32), False, 0, m["k"])
    s, rows = r.per_field_topk(torch.from_numpy(z["q"]).to(DEV), None, m["k"])
    s, rows = s.cpu().numpy(), rows.cpu().numpy()
    ref_s, ref_r = z["ref_retrieve_scores"], z["ref_retrieve_rows"]
    np.testing.assert_allclose(s, ref_s, rtol=2e-5, atol=2e-5 * np.abs(ref_s).max())
    mism = rows != ref_r
    for f, qi, j in np.argwhere(mism):                       # only (near-)ties may differ in order
        near = np.abs(ref_s[f, qi] - ref_s[f, qi, j]) <= 1e-5 * max(1.0, np.abs(ref_s[f, qi]).max())
        assert near.sum() > 1, (f, qi, j)


def test_dense_flat_index_api_matches_reference_types():
    from mfar_b200.data.index import DenseFlatIndex
    z, m = load(os.path.join(GOLDEN, "d768_dense_static.npz"))
    keys = [f"d{i}" for i in range(m["N"])]
    idx = DenseFlatIndex(None, z["fields"][0], keys, {k: i for i, k in enumerate(keys)}, device=DEV)
    hits = idx.retrieve_batch(z["q"], top_k=m["k"])
    assert len(hits) == m["Q"] and len(hits[0]) == m["k"]
    assert isinstance(hits[0][0][0], str) and isinstance(hits[0][0][1], float)
    assert [h[0] for h in hits[0]] == [f"d{r}" for r in z["ref_retrieve_rows"][0, 0]]
    cand = [keys[r] for r in z["cand_rows"]]
    sb = idx.score_batch(z["q"], cand).cpu().numpy()
    np.testing.assert_allclose(sb, z["ref_score_batch"][0], rtol=2e-5, atol=1e-4)
    with pytest.raises(KeyError):
        idx.score_batch(z["q"], ["nope"])
    single = idx.retrieve(z["q"][:1], 5)
    assert len(single) == 5
    idx.vectors = z["fields"][1]                              # rebinding re-packs (contrastive.py:493-494)
    assert [h[0] for h in idx.retrieve_batch(z["q"], m["k"])[1]] == [f"d{r}" for r in z["ref_retrieve_rows"][1, 1]]


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_score_candidates_vs_reference_score_batch(path):
    z, m = load(path)
    fields = [torch.from_numpy(z["fields"][f]) for f in range(m["Fd"])]
    sp = torch.from_numpy(z["sparse"]).to(DEV) if m["Fs"] else None
    F = m["Fd"] + m["Fs"]
    r = build(fields, np.ones((F, 1), np.float32), False, m["Fs"], m["k"])
    rows = torch.from_numpy(np.concatenate([z["cand_rows"], [-1]]))
    out = r.score_candidates(torch.from_numpy(z["q"]).to(DEV), rows, sp).cpu().numpy()
    np.testing.assert_allclose(out[: m["Fd"], :, :-1], z["ref_score_batch"], rtol=2e-5, atol=1e-4)
    assert (out[:, :, -1] == 0).all()
    if m["Fs"]:
        np.testing.assert_array_equal(out[m["Fd"]:], z["ref_sparse_score_batch"])


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_union_rescore_vs_reference_pipeline(path):
    z, m = load(path)
    fields = [torch.from_numpy(z["fields"][f]) for f in range(m["Fd"])]
    sp = torch.from_numpy(z["sparse"]).to(DEV) if m["Fs"] else None
    r = build(fields, z["W"], m["query_cond"], m["Fs"], m["k"])
    r.mask = torch.from_numpy(z["mask"]).to(DEV)
    q = torch.from_numpy(z["q"]).to(DEV)
    if bool(z["ref_union_raises"]):
        with pytest.raises(RuntimeError):
            r.union_rescore(q, q, sp)
        return
    vals, rows = r.union_rescore(q, q, sp)
    for i in range(m["Q"]):
        ref_v, ref_r = z["ref_union_vals"][i], z["ref_union_rows"][i]
        np.testing.assert_allclose(vals[i].cpu().numpy(), ref_v, rtol=2e-5, atol=1e-5)
        got_r = rows[i].cpu().numpy()
        for j in np.nonzero(got_r != ref_r)[0]:
            assert (np.abs(ref_v - ref_v[j]) <= 1e-5 * max(1.0, np.abs(ref_v).max())).sum() > 1


@pytest.mark.parametrize("shape", [(81, 5000, 768, 3, 2, 70, True, 100), (82, 3000, 256, 8, 0, 9, False, 100),
                                   (83, 2000, 128, 1, 3, 33, True, 50), (84, 900, 64, 0, 4, 5, False, 20),
                                   (85, 700, 64, 22, 22, 3, True, 20)], ids=lambda s: f"s{s[0]}")
def test_union_rescore_batch_on_device_vs_oracle_pipeline(shape):
    """The whole candidate stage of trec_eval_step (contrastive.py:676-696) in one launch for the batch
    (``mfar_union_rescore``) against the oracle's per-query restatement: same union sizes, same values, same rows up to
    near-ties; a masked field; more sparse than dense fields; sparse-only; 44 fields."""
    seed, N, d, Fd, Fs, Q, qc, k = shape
    fields, q, sp, W = synth(seed, N, d, Fd, Fs, Q, qc)
    r = build(fields, W, qc, Fs, k, n_docs=N)
    mask = torch.ones(Fd + Fs, 1)
    if Fd + Fs > 2:
        mask[1] = 0
        r.mask_field([1])
    qd = q.to(DEV)
    vals, rows, usize = r.union_rescore_batch(qd if Fd else None, qd, None if sp is None else sp.to(DEV), k,
                                              batch=Q)
    ref_v, ref_r = O.union_rescore(q, fields, None if sp is None else sp.float(), q, W, qc, mask, k)
    # union sizes: recompute from the oracle's per-field lists
    hits = [O.dense_retrieve_batch(q, f, k)[1] for f in fields] + \
           ([O.sparse_retrieve_batch(sp[:, j, :].float(), k)[1] for j in range(Fs)] if Fs else [])
    for i in range(Q):
        want_u = len(set().union(*[set(h[i].tolist()) for h in hits]))
        assert abs(int(usize[i]) - want_u) <= 2, (i, int(usize[i]), want_u)      # near-ties at a field's k-th place
        np.testing.assert_allclose(vals[i].cpu().numpy(), ref_v[i].numpy(), rtol=2e-5, atol=1e-5)
        got_r, want_r = rows[i].cpu().numpy(), np.asarray(ref_r[i])
        rv = ref_v[i].numpy()
        for j in np.nonzero(got_r != want_r)[0]:
            assert (np.abs(rv - rv[j]) <= 1e-5 * max(1.0, np.abs(rv).max())).sum() > 1, (i, j)
    lv, lr = r.union_rescore(qd if Fd else None, qd, None if sp is None else sp.to(DEV), k, batch=Q)
    assert len(lv) == Q and torch.equal(lv[0], vals[0]) and torch.equal(lr[-1], rows[-1])


def test_search_host_equals_device_search_and_counts_launches():
    fields, q, sp, W = synth(31, 1000, 768, 3, 2, 9, True)
    r = build(fields, W, True, 2, 100)
    s_dev, i_dev = r.search(q.to(DEV), q.to(DEV), sp.to(DEV))
    assert r.last_launches == 3                         # sparse pre-mix + scoring + merge
    qh = q.to(torch.bfloat16).pin_memory()
    s_h, i_h = r.search_host(qh, q.float().pin_memory(), sp.pin_memory())
    assert not s_h.is_cuda
    assert torch.equal(s_h, s_dev.cpu()) and torch.equal(i_h, i_dev.cpu())
    assert r.last_launches == 3                         # mixture weights + scoring (sparse gathered in its epilogue) + merge


@pytest.mark.parametrize("impl", ["tcgen05", "tcgen05_qs", "auto"])
@pytest.mark.parametrize("shape", [(71, 1111, 768, 8, 8, 3), (72, 3001, 256, 1, 2, 257), (73, 2000, 768, 22, 22, 64),
                                   (74, 129, 64, 2, 1, 17), (75, 5000, 128, 3, 5, 140), (76, 640, 64, 2, 3, 40)],
                         ids=lambda s: f"s{s[0]}")
def test_sparse_gather_fused_into_the_scoring_epilogue(shape, impl):
    """north_star (2): sparse score rows with a 32-byte aligned pitch are gathered and mixed inside the scoring
    epilogue - no pre-mix launch, no [Q,N] block (index.py:111-118 + contrastive.py:681-686 in one pass).  f16 and f32
    rows, ragged tails, single-field two-epilogue-set variant; agrees with the pre-mix path (unaligned pitch)."""
    seed, N, d, Fd, Fs, Q = shape
    fields, q, sp, W = synth(seed, N, d, Fd, Fs, Q, True)
    r = build(fields, W, True, Fs, 100, impl=impl)
    r.mask_field([Fd])                                   # a masked sparse field
    mask = torch.ones(Fd + Fs, 1)
    mask[Fd] = 0
    ref = O.exhaustive_scores(q, fields, sp.float(), O.mixture_weights(q, W, True), mask)
    ld = (N + 63) // 64 * 64
    qd = q.to(DEV)
    n_u = N if N % 16 else N + 1                         # a pitch that is NOT 32-byte aligned -> pre-mix kernel + base block
    unaligned = torch.zeros((Q, Fs, n_u), dtype=torch.float16, device=DEV)
    unaligned[:, :, :N] = sp.to(DEV)
    s0, i0 = r.search(qd, qd, unaligned)
    assert r.last_launches == 3                          # pre-mix + scoring + merge
    for dtype in (torch.float16, torch.float32):
        padded = torch.zeros((Q, Fs, ld), dtype=dtype, device=DEV)
        padded[:, :, :N] = sp.to(DEV)
        s1, i1 = r.search(qd, qd, padded)
        assert r.last_launches == 2                      # scoring + merge
        assert_topk_parity(s1.cpu().numpy(), i1.cpu().numpy(), ref.numpy(), 100)
        # same result as the pre-mix path up to fp32 summation order (the query-stationary epilogue interleaves the
        # sparse and dense terms)
        assert_same_topk_up_to_ties(s1.cpu(), i1.cpu(), s0.cpu(), i0.cpu())


@pytest.mark.parametrize("impl", IMPLS)
def test_virtual_shards_merge_equals_single_shard(impl):
    """Shard-merge associativity: 1 vs 2/4/8 doc-range shards (run sequentially on one GPU, global ids,
    keys merged by mfar_topk_merge) give bit-identical results."""
    from mfar_b200.dist import merge_keys, shard_range
    fields, q, sp, W = synth(41, 4000, 768, 3, 1, 5, True)
    k = 100

    def pitched(x):                                  # 128-byte row pitch: every shard takes the fused sparse gather
        out = torch.zeros((x.shape[0], x.shape[1], (x.shape[2] + 63) // 64 * 64), dtype=x.dtype, device=DEV)
        out[:, :, :x.shape[2]] = x
        return out
    full = build(fields, W, True, 1, k, impl=impl)
    s0, i0, k0 = full.search(q.to(DEV), q.to(DEV), pitched(sp), return_keys=True)
    for R in (2, 4, 8):
        keys = []
        for rank in range(R):
            lo, hi = shard_range(4000, rank, R)
            sh = build([f[lo:hi] for f in fields], W, True, 1, k, doc_id_base=lo, impl=impl)
            _, _, kk = sh.search(q.to(DEV), q.to(DEV), pitched(sp[:, :, lo:hi]), return_keys=True)
            keys.append(kk)
        s, i = merge_keys(torch.stack(keys), k)
        assert torch.equal(i, i0) and torch.equal(s, s0), R


@pytest.mark.parametrize("impl", IMPLS)
def test_corpus_windows_with_moved_boundaries_equal_the_unsharded_search(impl):
    """Tunable shard boundaries (dist.held_ranges / rebalanced_boundaries, PackedCorpus.window): every virtual rank packs
    its range plus a margin of its neighbours' docs, searches a zero-copy WINDOW of it, the boundaries move, and the
    merged result stays bit-identical to the unsharded search - before and after the move."""
    MultiFieldRetriever, PackedCorpus, LinearWeights = _mods()
    from mfar_b200.dist import held_ranges, merge_keys, rebalanced_boundaries, weighted_shard_ranges
    N, R, k, margin = 6000, 3, 100, 384
    fields, q, _, W = synth(43, N, 256, 2, 0, 40, True)
    full = build(fields, W, True, 0, k, impl=impl)
    s0, i0, _ = full.search(q.to(DEV), q.to(DEV), None, return_keys=True)
    base = [r[0] for r in weighted_shard_ranges(N, [1.0] * R)] + [N]
    held = held_ranges(base, margin, N)
    packed = [PackedCorpus.from_fields([f[lo:hi] for f in fields], DEV) for lo, hi in held]
    layer = full.mixture
    cuts = list(base)
    for step_ms in (None, [1.0, 1.3, 0.9], [1.2, 1.0, 1.0]):
        if step_ms is not None:
            cuts = rebalanced_boundaries(cuts, step_ms, base, margin)
            assert cuts != base and all(abs(c - b) <= margin and c % 128 == 0 for c, b in zip(cuts[1:-1], base[1:-1]))
        keys = []
        for r in range(R):
            lo, hi = cuts[r], cuts[r + 1]
            win = packed[r].window(lo - held[r][0], hi - lo)
            assert win.data.data_ptr() == packed[r].data.data_ptr() + \
                (lo - held[r][0]) // 128 * 2 * 128 * win.dim_pad * 2          # a pointer offset, not a copy
            sh = MultiFieldRetriever(win, layer, top_k=k, doc_id_base=lo, impl=impl, n_docs=hi - lo, device=DEV)
            keys.append(sh.search(q.to(DEV), q.to(DEV), None, return_keys=True)[2])
        s, i = merge_keys(torch.stack(keys), k)
        assert torch.equal(i, i0) and torch.equal(s, s0), cuts
    with pytest.raises(ValueError):
        packed[0].window(64, 100)                                              # not on a tile boundary


@pytest.mark.parametrize("impl", IMPLS)
def test_sparse_coo_input_equals_dense_input_and_oracle(impl, tmp_path):
    """Sparse scores given in the reference's precomputed-BM25 file layout (int32 (qid, doc) pairs + f16 values per
    field, precompute_bm25s_scores.py:21-30) vs the same scores as a dense [Q,Fs,N] tensor vs the oracle; a sharded
    retriever must skip the pairs of other shards."""
    from mfar_b200.data.typedef import Field, FieldType
    from mfar_b200.modeling.util import PrecomputedSparseScores
    seed, N, d, Fd, Fs, Q, k = 41, 1500, 128, 2, 3, 7, 50
    fields, q, sp, W = synth(seed, N, d, Fd, Fs, Q, True)
    qids = [1000 + 7 * i for i in range(Q)]
    finfo = {f"s{j}_sparse": Field(f"s{j}_sparse", f"s{j}", FieldType.SPARSE) for j in range(Fs)}
    for j, fk in enumerate(finfo):                                     # write the files the reference would
        nz = torch.nonzero(sp[:, j, :])
        order = torch.randperm(len(nz), generator=torch.Generator().manual_seed(j))
        nz = nz[order]
        keys = np.stack([np.array(qids)[nz[:, 0].numpy()], nz[:, 1].numpy()], axis=1).astype(np.int32)
        np.save(tmp_path / f"{fk}_keys_bm25.npy", keys)
        np.save(tmp_path / f"{fk}_vals_bm25.npy", sp[nz[:, 0], j, nz[:, 1]].numpy().astype(np.float16))
    store = PrecomputedSparseScores.load(str(tmp_path), finfo)
    assert store.lookup("s1_sparse", qids[2], int(torch.nonzero(sp[2, 1])[0])) == float(sp[2, 1, torch.nonzero(sp[2, 1])[0]])
    assert store.lookup("s1_sparse", qids[2], int(torch.nonzero(sp[2, 1] == 0)[0])) == 0.0
    coo = store.batch(qids, DEV)
    if impl == "simt" or Fd:
        r = build(fields, W, True, Fs, k, impl=impl)
        s_coo, i_coo = r.search(q.to(DEV), q.to(DEV), sparse_coo=coo)
        s_dense, i_dense = r.search(q.to(DEV), q.to(DEV), sp.to(DEV))
        torch.testing.assert_close(s_coo, s_dense, rtol=1e-6, atol=1e-5)
        assert_same_topk_up_to_ties(s_coo.cpu(), i_coo.cpu(), s_dense.cpu(), i_dense.cpu())
        ref = O.exhaustive_scores(q, fields, sp.float(), O.mixture_weights(q, W, True))
        assert_topk_parity(s_coo.cpu().numpy(), i_coo.cpu().numpy(), ref.numpy(), k)
        lo, hi = 512, 1100                                             # a shard: global doc rows [lo, hi)
        sh = build([f[lo:hi] for f in fields], W, True, Fs, k, doc_id_base=lo, impl=impl)
        s_sh, i_sh = sh.search(q.to(DEV), q.to(DEV), sparse_coo=coo)
        assert_topk_parity(s_sh.cpu().numpy(), i_sh.cpu().numpy(), ref[:, lo:hi].numpy(), k, id_offset=lo)


def test_mask_sweep_in_one_pass_equals_mask_field_loop():
    """mask_fields.py:142-170 (baseline, each field, all sparse, all dense, each name) as extra weight rows of one
    fused pass vs. the reference's procedure: mask_field(idx) + a full search per masking; also vs the oracle."""
    from mfar_b200.data.schema import resolve_fields
    finfo = resolve_fields("all_dense,all_sparse", "mag")                      # 5 dense + 5 sparse
    plan = _mods()[0].mask_sweep_plan(finfo)
    assert [p[0] for p in plan][:2] == ["baseline", f"field:{next(iter(finfo))}"] and len(plan) == 1 + 10 + 2 + 5
    Fd = Fs = 5
    fields, q, sp, W = synth(51, 3000, 768, Fd, Fs, 9, True)
    r = build(fields, W, True, Fs, 100)
    S, I = r.search_mask_sweep(q.to(DEV), [p[1] for p in plan], q.to(DEV), sp.to(DEV), max_rows=64)
    w = O.mixture_weights(q, W, True)
    for m, (label, idx) in enumerate(plan):
        r.mask_field(idx)
        s1, i1 = r.search(q.to(DEV), q.to(DEV), sp.to(DEV))
        torch.testing.assert_close(S[m], s1, rtol=2e-5, atol=1e-4)
        assert_same_topk_up_to_ties(S[m].cpu(), I[m].cpu(), s1.cpu(), i1.cpu())
        mask = torch.ones(Fd + Fs, 1)
        mask[idx] = 0
        ref = O.exhaustive_scores(q, fields, sp.float(), w, mask)
        assert_topk_parity(S[m].cpu().numpy(), I[m].cpu().numpy(), ref.numpy(), 100)
    r.mask_field([])


def test_peer_exchange_merge_virtual_ranks():
    """The fused NVLink exchange+merge kernel with R "virtual ranks" on one device: R exchange buffers, R concurrent
    streams, each rank pushing into all buffers and spinning on its own flags.  Three epochs (both parities and a
    buffer reuse).  Must equal a single merge of the concatenated lists."""
    from mfar_b200.dist import PeerExchange, encode_keys, merge_keys
    R, Q, k = 4, 9, 100
    n = PeerExchange.buffer_bytes(R, 16, 128)
    bufs = [torch.zeros(n, dtype=torch.uint8, device=DEV) for _ in range(R)]
    ex = [PeerExchange(16, 128, peer_buffers=bufs, rank=r, world=R) for r in range(R)]
    streams = [torch.cuda.Stream() for _ in range(R)]
    g = np.random.RandomState(5)
    for epoch in range(3):
        scores = g.standard_normal((R, Q, k)).astype(np.float32) * 10
        ids = np.stack([g.permutation(100000)[: Q * k].reshape(Q, k) + 100000 * r for r in range(R)])
        keys = torch.from_numpy(encode_keys(scores, ids).view(np.int64)).to(DEV)         # [R,Q,k]
        want_s, want_i = merge_keys(keys, k)
        torch.cuda.synchronize()
        outs = []
        for r in range(R):
            with torch.cuda.stream(streams[r]):
                outs.append(ex[r].merge(keys[r], k))
        torch.cuda.synchronize()
        for s_r, i_r in outs:
            assert torch.equal(s_r, want_s) and torch.equal(i_r, want_i)


def test_pipelined_exchange_virtual_ranks():
    """push / wait_merge(lag): a step pushes its keys and merges the PREVIOUS step's (four rotating slots).  R virtual
    ranks on one device, 7 epochs incl. changes of the batch size: every wait_merge(1) returns the merge of the previous
    epoch's lists (empty rows for queries the previous epoch did not push, (-inf, -1) rows at the very first call),
    wait_merge(0) at the end the last epoch's - all equal to mfar_topk_merge of the same lists."""
    from mfar_b200.dist import PeerExchange, encode_keys, merge_keys
    R, k = 4, 100
    n = PeerExchange.buffer_bytes(R, 16, 128)
    bufs = [torch.zeros(n, dtype=torch.uint8, device=DEV) for _ in range(R)]
    ex = [PeerExchange(16, 128, peer_buffers=bufs, rank=r, world=R) for r in range(R)]
    streams = [torch.cuda.Stream() for _ in range(R)]
    g = np.random.RandomState(9)
    want_prev = None
    for Q in (11, 11, 5, 5, 11, 11, 11):
        scores = g.standard_normal((R, Q, k)).astype(np.float32) * 10
        ids = np.stack([g.permutation(100000)[: Q * k].reshape(Q, k) + 100000 * r for r in range(R)])
        keys = torch.from_numpy(encode_keys(scores, ids).view(np.int64)).to(DEV)         # [R,Q,k]
        want = merge_keys(keys, k)
        torch.cuda.synchronize()
        outs = []
        for r in range(R):
            with torch.cuda.stream(streams[r]):
                ex[r].push(keys[r])
                outs.append(ex[r].wait_merge(k, lag=1))
        torch.cuda.synchronize()
        for s_r, i_r in outs:
            assert s_r.shape == (Q, k)
            n_prev = 0 if want_prev is None else min(Q, want_prev[0].shape[0])
            assert torch.equal(s_r[:n_prev], want_prev[0][:n_prev]) if n_prev else True
            assert torch.equal(i_r[:n_prev], want_prev[1][:n_prev]) if n_prev else True
            assert torch.isinf(s_r[n_prev:]).all() and (i_r[n_prev:] == -1).all()
        want_prev = want
    outs = []
    for r in range(R):
        with torch.cuda.stream(streams[r]):
            outs.append(ex[r].wait_merge(k, lag=0))
    torch.cuda.synchronize()
    for s_r, i_r in outs:
        assert torch.equal(s_r, want_prev[0]) and torch.equal(i_r, want_prev[1])


def test_topk_edge_cases():
    fields, q, _, W = synth(51, 300, 64, 2, 0, 2, False)
    r = build(fields, W, False, 0, 100)
    with pytest.raises(RuntimeError):                   # reference: torch.topk raises when k > N
        r.search(q.to(DEV), None, None, top_k=301)
    # all-equal scores: deterministic tie-break = lowest doc ids first
    zeros = [torch.zeros(300, 64)]
    rz = build(zeros, np.ones((1, 1), np.float32), False, 0, 10)
    s, i = rz.search(q.to(DEV))
    assert (s == 0).all() and i.cpu().tolist() == [list(range(10))] * 2
    # masks: masking every field but one == searching that field alone (weights not renormalised)
    r.mask_field([0])
    s1, i1 = r.search(q.to(DEV), top_k=20)
    w = O.mixture_weights(None, W, False)
    ref = O.exhaustive_scores(q, fields, None, w, torch.tensor([[0.0], [1.0]]))
    assert_topk_parity(s1.cpu().numpy(), i1.cpu().numpy(), ref.numpy(), 20)


def test_trec_eval_step_writes_qres_lines():
    fields, q, _, W = synth(61, 400, 64, 2, 0, 3, True)
    r = build(fields, W, True, 0, 100)
    r.numeric_ids_to_keys = [f"doc{i}" for i in range(400)]
    buf = io.StringIO()
    r.trec_eval_step(["qa", "qb", "qc"], q.to(DEV), buf, q_emb=q.to(DEV))
    lines = buf.getvalue().strip().split("\n")
    assert len(lines) == 300
    qid, it, doc, rank, sim, run = lines[0].split("\t")
    assert qid == "qa" and it == "0" and doc.startswith("doc") and run == "0"
    sims = [float(l.split("\t")[4]) for l in lines[:100]]
    assert sims == sorted(sims, reverse=True)
