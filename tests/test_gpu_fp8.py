"""The E4M3 corpus (``PackedCorpus(dtype="e4m3")``) on the GPU.

1. The pack kernel stores the oracle's payload bytes and scales bit for bit (``e4m3_oracle.quantize_rows_e4m3``), for
   docs and queries, with and without the cosine normalisation, whatever the slab order; unpack is exact.
2. On inputs whose scores are exact in fp32 whatever the summation order (small integers, exact in E4M3, and mixture
   weights 1/F), every scoring path equals both the oracle's closed form and the bf16 search of the dequantized corpus
   element for element: ids, scores and the (score desc, doc id asc) tie order.
3. At corpus scale (threshold seeding, list overflow) the E4M3 search is ranked against ``tests/checker.py`` on the
   dequantized bf16 copy with the near-tie rule of ``tests/parity.py`` - the bf16 bar, not a wider one.
"""
import gc

import numpy as np
import pytest
import torch

import e4m3_oracle as E
import mfar_oracle as O
from checker import Fp32Checker, assert_topk_parity_at_scale
from parity import assert_topk_parity

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _retriever(fields, Fs=0, dtype="e4m3", top_k=100, doc_id_base=0, sparse_indices=None):
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    F = len(fields) + (len(sparse_indices) if sparse_indices else Fs)
    layer = LinearWeights(F, 1)                          # softmax of zeros: every weight is exactly 1/F
    with torch.no_grad():
        layer.weight.zero_()
    pc = PackedCorpus.from_fields(fields, DEV, dtype=dtype)
    return MultiFieldRetriever(pc, layer.to(DEV), n_sparse=Fs, top_k=top_k, doc_id_base=doc_id_base,
                               sparse_indices=sparse_indices)


def _dequantized_twin(r):
    """The bf16 retriever over the dequantized copy of an E4M3 retriever's corpus (exact: E4M3 x 2^e is a bf16 value)."""
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    pc = r.corpus
    twin = PackedCorpus(pc.n_docs, pc.n_fields, pc.dim, DEV)
    for f in range(pc.n_fields):
        twin.load_rows(f, 0, pc.unpack_field(f))
    t = MultiFieldRetriever(twin, r.mixture, n_sparse=r.n_sparse, top_k=r.top_k, doc_id_base=r.doc_id_base,
                            impl=r.impl)
    t.bm25 = r.bm25
    return t


def _dequantize_queries(pc, q):
    payload, scales = pc.prepare_queries(q)
    return (payload.view(torch.float8_e4m3fn).float() * scales[:, None])[:, : pc.dim]


def _int_case(N, Fd, D, Q, seed, Fs=0):
    """Doc coordinates 0..15 (many exact duplicates across tiles), query coefficients -15..15 (query 0 is all zeros:
    every doc ties), sparse scores 0..15 in f16: every score is an integer well inside fp32's exact range."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 16, size=(97, D))
    fields = []
    for _ in range(Fd):
        x = rng.integers(0, 16, size=(N, D))
        dup = rng.random(N) < 0.3
        x[dup] = base[rng.integers(0, 97, size=int(dup.sum()))]
        fields.append(torch.from_numpy(x.astype(np.float32)))
    q = torch.from_numpy(rng.integers(-15, 16, size=(Q, D)).astype(np.float32))
    q[0] = 0
    sp = None
    if Fs:
        sp = torch.from_numpy(rng.integers(0, 16, size=(Q, Fs, N)) * (rng.random((Q, Fs, N)) < 0.3)).half()
    return fields, q, sp


def _oracle_topk(fields, q, sp, k, base=0):
    F = len(fields) + (0 if sp is None else sp.shape[1])
    w = torch.full((1, F), 1.0 / F)
    s, i = O.topk_sorted(O.exhaustive_scores(q, fields, None if sp is None else sp.float(), w), k)
    return s, i + base


def _eq(got, want, what):
    s, i = got
    ws, wi = want
    s, i = s.cpu(), i.cpu()
    assert torch.equal(i, wi.cpu()), f"{what}: ids differ in {(i != wi.cpu()).any(1).sum().item()} queries"
    assert torch.equal(s, ws.cpu()), f"{what}: scores differ"


# ---------------------------------------------------------------------------------------------------------- 1. pack
def _edge_rows(D):
    rng = np.random.default_rng(3)
    rows = [np.zeros(D), -np.zeros(D), np.full(D, 448.0), np.full(D, 449.0), np.full(D, 2.0 ** -140),
            np.full(D, 3.3e38), np.r_[np.nan, np.ones(D - 1)], np.r_[np.ones(D - 1), -np.inf],
            np.r_[1e-30 * rng.standard_normal(D - 1), 0.0], np.r_[2.0 ** -120, np.full(D - 1, 2.0 ** -125)],
            1.0625 * np.sign(rng.standard_normal(D)), 1e19 * rng.standard_normal(D)]
    return np.stack(rows).astype(np.float32)


@pytest.mark.parametrize("normalize", [False, True])
@pytest.mark.parametrize("src", ["f32", "bf16"])
def test_pack_matches_oracle_bit_for_bit(normalize, src):
    from mfar_b200.modeling.retrieval import PackedCorpus
    D, N, F = 200, 1000, 3
    rng = np.random.default_rng(11)
    x = (rng.standard_normal((F, N, D)) * np.exp(rng.uniform(-30, 30, (F, N, 1)))).astype(np.float32)
    e = _edge_rows(D)
    x[1, 500:500 + len(e)] = e
    xt = torch.from_numpy(x)
    if src == "bf16":
        xt = xt.to(torch.bfloat16)
    pc = PackedCorpus(N, F, D, DEV, normalize=normalize, dtype="e4m3")
    assert pc.data.dtype == torch.uint8 and pc.dim_pad == 256
    slabs = [(f, lo) for f in range(F) for lo in range(0, N, 128 * 3)]
    for j in rng.permutation(len(slabs)):                   # slabs in any order
        f, lo = slabs[j]
        pc.load_rows(f, lo, xt[f, lo:lo + 384])
    tiles = (N + 127) // 128
    payload = pc.data.view(tiles, F, 128, pc.dim_pad).cpu().numpy()
    scales = pc.scales.view(tiles, F, 128).cpu().numpy()
    for f in range(F):
        want_p, want_s = E.quantize_rows_e4m3(xt[f].float(), normalize=normalize)
        got_p = payload[:, f].reshape(-1, pc.dim_pad)
        got_s = scales[:, f].reshape(-1)
        assert np.array_equal(got_p[:N, :D], want_p), f"field {f} payload"
        assert not got_p[:, D:].any() and not got_p[N:].any()
        assert np.array_equal(got_s[:N].view(np.uint32), want_s.view(np.uint32)), f"field {f} scales"
        assert (got_s[N:] == 1.0).all()
        got_d = pc.unpack_field(f).cpu().numpy()
        want_d = E.dequantize_rows_e4m3(want_p, want_s)
        assert np.array_equal(np.isnan(got_d), np.isnan(want_d))
        assert np.array_equal(np.nan_to_num(got_d), np.nan_to_num(want_d))
    # queries: the same kernel, the same rule
    qp, qs = pc.prepare_queries(xt[1, 490:520])
    want_p, want_s = E.quantize_rows_e4m3(xt[1, 490:520].float(), normalize=normalize)
    assert qp.dtype == torch.uint8 and qp.shape == (30, pc.dim_pad)
    assert np.array_equal(qp[:, :D].cpu().numpy(), want_p)
    assert np.array_equal(np.nan_to_num(qs.cpu().numpy(), nan=-1), np.nan_to_num(want_s, nan=-1))


# --------------------------------------------------------------------------------------------------- 2. exact search
_small = {}


def _small_case():
    if not _small:
        fields, q, sp = _int_case(5000, 2, 128, 130, seed=21, Fs=2)
        r = _retriever(fields, Fs=2)
        _small.update(fields=fields, q=q, sp=sp, r=r, twin=_dequantized_twin(r))
    return _small


@pytest.mark.parametrize("impl", ["simt", "tcgen05", "auto"])
@pytest.mark.parametrize("Q", [1, 20, 64, 130])
def test_search_exact(impl, Q):
    c = _small_case()
    fields, q = c["fields"], c["q"][:Q]
    rd = _retriever(fields)                                  # dense only (F = 2)
    want = _oracle_topk(fields, q, None, 100)
    _eq(rd.search(q.to(DEV), impl=impl), want, f"e4m3 {impl} Q={Q}")
    _eq(_dequantized_twin(rd).search(q.to(DEV), impl=impl), want, f"bf16 twin {impl} Q={Q}")


def test_query_stationary_kernel_refuses_e4m3():
    c = _small_case()
    with pytest.raises(RuntimeError, match="shape"):
        c["r"].search(c["q"][:100].to(DEV), sparse=c["sp"][:100].to(DEV), impl="tcgen05_qs")
    for call in (lambda: c["r"].union_rescore(c["q"][:4].to(DEV), sparse=c["sp"][:4].to(DEV)),
                 lambda: c["r"].search_host(torch.zeros((1, 128), dtype=torch.bfloat16))):
        with pytest.raises(ValueError, match="E4M3"):
            call()


@pytest.mark.parametrize("layout", ["fused", "unaligned", "coo"])
@pytest.mark.parametrize("impl", ["simt", "tcgen05", "auto"])
def test_sparse_inputs_exact(layout, impl):
    c = _small_case()
    r, q, sp = c["r"], c["q"].to(DEV), c["sp"]
    N = sp.shape[2]
    want = _oracle_topk(c["fields"], c["q"], sp, 100)
    if layout == "coo":
        nz = sp.nonzero()                                    # (query, field, doc), field-major below
        order = torch.argsort(nz[:, 1] * (1 << 40) + nz[:, 0] * (1 << 20) + nz[:, 2])
        nz = nz[order]
        keys = torch.stack([nz[:, 0], nz[:, 2]], 1).int().to(DEV)
        vals = sp[nz[:, 0], nz[:, 1], nz[:, 2]].to(DEV)
        off = [0] + torch.bincount(nz[:, 1], minlength=2).cumsum(0).tolist()
        got = r.search(q, sparse_coo=(keys, vals, off), impl=impl)
        twin = c["twin"].search(q, sparse_coo=(keys, vals, off), impl=impl)
    else:
        ld = 5056 if layout == "fused" else 5003           # 32-byte rows are gathered in the epilogue, others pre-mixed
        buf = torch.zeros((sp.shape[0], 2, ld), dtype=torch.float16, device=DEV)
        buf[:, :, :N] = sp.to(DEV)
        got = r.search(q, sparse=buf, impl=impl)
        twin = c["twin"].search(q, sparse=buf, impl=impl)
    _eq(got, want, f"{layout} {impl}")
    _eq(twin, want, f"{layout} {impl} bf16 twin")


def test_bm25_tokens_match_dequantized_bf16():
    from mfar_b200.data.bm25 import DeviceBM25
    c = _small_case()
    rng = np.random.default_rng(4)
    V, N, Q = 300, 5000, 40
    corpora = [[rng.integers(0, V, size=rng.integers(1, 12)).tolist() for _ in range(N)] for _ in range(2)]
    tokens = [[rng.integers(0, V, size=4).tolist() for _ in range(Q)] for _ in range(2)]
    bm = [DeviceBM25(device=DEV).index(cc, vocab=V) for cc in corpora]
    r = _retriever(c["fields"], sparse_indices=bm)
    twin = _dequantized_twin(r)
    q = c["q"][:Q].to(DEV)
    s, i = r.search(q, sparse_tokens=tokens)
    ts, ti = twin.search(q, sparse_tokens=tokens)
    spb = r.bm25_field_scores(tokens, Q)[:, :, :N].float().cpu()
    ref = O.exhaustive_scores(c["q"][:Q], c["fields"], spb, torch.full((1, 4), 0.25))
    for got in ((s, i), (ts, ti)):                           # fp32 atomics order the BM25 sums: the near-tie rule
        assert_topk_parity(got[0].cpu().numpy(), got[1].cpu().numpy(), ref.numpy(), 100, rtol=1e-4, tie_rel=1e-4)


def test_per_field_mask_sweep_candidates_exact():
    c = _small_case()
    r, twin, q, sp = c["r"], c["twin"], c["q"][:33].to(DEV), c["sp"][:33].to(DEV)
    a, b = r.per_field_topk(q, sp), twin.per_field_topk(q, sp)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for f in range(2):                                       # the dense fields against the reference's running top-k
        ws, wi = O.dense_retrieve_batch(c["q"][:33], c["fields"][f], 100)
        assert torch.equal(a[0][f].cpu(), ws)
    sets = [[], [0], [1], [2, 3], [0, 2]]
    a, b = r.search_mask_sweep(q, sets, sparse=sp, max_rows=70), twin.search_mask_sweep(q, sets, sparse=sp, max_rows=70)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    rows = torch.tensor([0, 4999, 128, -1, 77, 3000], device=DEV)
    got, want = r.score_candidates(q, rows, sparse=sp), twin.score_candidates(q, rows, sparse=sp)
    assert torch.equal(got, want)
    dense = torch.stack([c["q"][:33] @ f_[rows.clamp(min=0).cpu()].t() for f_ in c["fields"]])
    dense[:, :, 3] = 0
    assert torch.equal(got[:2].cpu(), dense)


def test_window_shards_graph_and_batch_independence():
    from mfar_b200.dist import merge_keys
    from mfar_b200.modeling.retrieval import GraphedSearch, MultiFieldRetriever
    c = _small_case()
    fields = c["fields"]
    r = _retriever(fields)
    q = c["q"][:17].to(DEV)
    s, i, keys = r.search(q, return_keys=True)
    _eq((s, i), _oracle_topk(fields, c["q"][:17], None, 100), "unsharded")
    # every query alone
    for j in (0, 5, 16):
        sj, ij = r.search(q[j:j + 1])
        assert torch.equal(sj, s[j:j + 1]) and torch.equal(ij, i[j:j + 1])
    # doc-range windows (pointer offsets of payload AND scales) with global ids, merged
    cuts = [0, 128 * 13, 128 * 30, 5000]
    parts = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        sh = MultiFieldRetriever(r.corpus.window(lo, hi - lo), r.mixture, top_k=100, doc_id_base=lo)
        got = sh.search(q, return_keys=True)
        _eq(got[:2], _oracle_topk([f_[lo:hi] for f_ in fields], c["q"][:17], None, 100, base=lo), f"window [{lo},{hi})")
        parts.append(got[2])
    keys_parts = torch.stack(parts)
    sm, im = merge_keys(keys_parts, 100)
    assert torch.equal(sm, s) and torch.equal(im, i)
    # the quantization of the queries is captured in the graph
    g = GraphedSearch(r, 17)
    for salt in (0, 1):
        qq = q.flip(0) if salt else q
        gs, gi = g(qq)
        es, ei = r.search(qq)
        assert torch.equal(gs, es) and torch.equal(gi, ei)


def test_nan_rows_rank_first():
    c = _small_case()
    fields = [f_.clone() for f_ in c["fields"]]
    nan_docs = [7, 300, 4000]
    fields[1][nan_docs, 3] = float("nan")
    fields[0][1234, 0] = float("inf")
    r = _retriever(fields)
    q = c["q"][1:9].to(DEV)
    for impl in ("simt", "tcgen05", "auto"):
        s, i = r.search(q, impl=impl)
        assert torch.isnan(s[:, :4]).all() and not torch.isnan(s[:, 4:]).any()
        assert (i[:, :4].cpu() == torch.tensor([7, 300, 1234, 4000])).all()


# ---------------------------------------------------------------------------------------------------- 3. at scale
SCALE = {  # name: (n_docs, n_dense, n_sparse, doc_id_base, seed, batches)
    "c4_amazon_hybrid": (957_192, 8, 8, 0, 103, (64, 512)),
    "c5_shard_of_8": (1_250_000, 8, 0, 3_750_000, 104, (1, 64, 128, 512)),
}
SCALE_RUNS = [(n, b) for n, v in SCALE.items() for b in v[5]]
_big = {}


def _scale_case(name):
    if name in _big:
        return _big[name]
    _big.clear()
    gc.collect()
    torch.cuda.empty_cache()
    from mfar_b200 import synth as S
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    n, Fd, Fs, base, seed, batches = SCALE[name]
    D, Qmax, F = 768, max(batches), Fd + Fs
    pc = PackedCorpus(n, Fd, D, DEV, dtype="e4m3")
    S.fill_packed_corpus(pc, seed=seed)
    layer = LinearWeights(D, F, query_cond=True)
    with torch.no_grad():
        layer.weight.copy_(S.make_mixture(D, F, seed + 2))
    r = MultiFieldRetriever(pc, layer.to(DEV), n_sparse=Fs, top_k=100, doc_id_base=base)
    q = S.make_queries(Qmax, D, S.corpus_mean(D, seed, DEV), seed + 1, DEV)
    sp = None
    if Fs:
        sp = torch.zeros((Qmax, Fs, (n + 63) // 64 * 64), dtype=torch.float16, device=DEV)
        for q0 in range(0, Qmax, 32):
            sp[q0:q0 + 32, :, :n] = S.make_sparse(min(32, Qmax - q0), Fs, n, seed + 3 + q0, DEV)
    twin = _dequantized_twin(r).corpus
    qd = _dequantize_queries(pc, q)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    w = torch.softmax(q.float() @ layer.weight.detach().float().to(DEV), dim=1).contiguous()
    torch.backends.cuda.matmul.allow_tf32 = prev
    chk = Fp32Checker(twin, doc_id_base=base)
    ref_s, ref_i = chk.topk(qd, w, 100, sparse=sp, slack=64)
    _big[name] = dict(r=r, q=q, qd=qd, w=w, sp=sp, chk=chk, ref_s=ref_s, ref_i=ref_i, n=n, base=base)
    return _big[name]


@pytest.mark.parametrize("case,batch", SCALE_RUNS, ids=[f"{c}-Q{b}" for c, b in SCALE_RUNS])
def test_ranked_against_fp32_checker_at_scale(case, batch):
    c = _scale_case(case)
    sp = None if c["sp"] is None else c["sp"][:batch]
    q = c["q"][:batch]
    s, i = c["r"].search(q, q.float(), sp)
    torch.cuda.synchronize()
    resc = c["chk"].rescore(c["qd"][:batch], c["w"][:batch], i, sparse=sp)
    assert_topk_parity_at_scale(s, i, c["ref_s"][:batch], c["ref_i"][:batch], resc, 100, c["n"], c["base"],
                                what=f"e4m3 {case} Q={batch}")
    # the answers themselves are scored right: score_candidates of the returned rows, mixed, is the returned score
    if sp is None:
        m = min(4, batch)
        per_field = c["r"].score_candidates(q[:m], (i[:m] - c["base"]).reshape(-1))        # [F, m, m*100]
        mixed = torch.einsum("fqc,qf->qc", per_field, c["w"][:m]).view(m, m, 100)
        got = torch.stack([mixed[j, j] for j in range(m)])
        assert torch.allclose(got, s[:m], rtol=2e-5, atol=1e-5)


def test_zz_release_hbm():
    _small.clear()
    _big.clear()
    gc.collect()
    torch.cuda.empty_cache()
