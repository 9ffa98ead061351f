"""Exact top-k under ties: every scoring path against a closed-form answer, compared with ``torch.equal``.

The parity tests elsewhere accept any order and any membership inside a near-tie group, and their inputs are
continuous, so exact ties at rank k never occur there.  Here the inputs of tests/exact_topk.py make every mixture score
an exact fp32 integer (or an exact quarter / half of one), so the correct answer is the (score desc, doc id asc) order
that ``MultiFieldRetriever.search`` and ``DeviceBM25.retrieve`` document, and any other subset or order of a tie group
is a failure.  Each query of a batch takes one (pattern, sign), so one launch mixes tie groups at rank k across every
CTA, runs of duplicates across tiles and shard cuts, ascending scores (a compaction every tile), all-equal rows (the
exact-sort fallback of ``warp_select_keys``, the streaming path of the merge) and a tie-free control.

The large cases assert ``last_launches`` so that each provably ran the threshold-seeding levels it targets
(csrc/capi.cu: every prefix level adds 4 launches).
"""
import gc

import numpy as np
import pytest
import torch

import exact_topk as X

pytestmark = pytest.mark.gpu

DEV = "cuda"
KS = (1, 2, 100, 127, 128)
QS = (1, 16, 17, 32, 33, 64, 65, 128, 129, 257, 384, 512)
IMPLS = ("simt", "tcgen05", "tcgen05_qs", "auto")
TOP = 2 ** 32

# name: (N, dim, dense fields, sparse fields, doc_id_base)
CORPORA = {
    "s129": (129, 768, 1, 0, TOP - 129),
    "s4097": (4097, 768, 2, 2, TOP - 4097),
    "s4097_d64": (4097, 64, 4, 0, TOP - 4097),
    "m330k": (330_001, 768, 2, 2, TOP - 330_001),
    "l4m": (4_000_001, 64, 1, 0, TOP - 4_000_001),
}

_cache = {}


def _free():
    _cache.clear()
    gc.collect()
    torch.cuda.empty_cache()


def _sparse_rows(N, Fs):
    """int64 [Fs, N]: per-field sparse scores (f16-exact integers <= 2048), the same for every query."""
    n = np.arange(N, dtype=np.int64)
    rows = [(n // 7) % 11 * 64, np.where(n % 1009 == 5, 2048, (n * 13) % 17)]
    return np.stack(rows[:Fs]) if Fs else np.zeros((0, N), dtype=np.int64)


def _corpus(name):
    if name in _cache:
        return _cache[name]
    if name in ("m330k", "l4m"):                      # one large corpus at a time
        for other in ("m330k", "l4m"):
            _cache.pop(other, None)
        gc.collect()
        torch.cuda.empty_cache()
    from mfar_b200.modeling.retrieval import PackedCorpus
    N, dim, Fd, Fs, base = CORPORA[name]
    pc = PackedCorpus(N, Fd, dim, DEV)
    docs = X.doc_matrix(N, dim)
    for lo in range(0, N, 1 << 18):
        hi = min(N, lo + (1 << 18))
        rows = torch.from_numpy(docs[lo:hi]).to(DEV).to(torch.bfloat16)
        for f in range(Fd):
            pc.load_rows(f, lo, rows)
    c = dict(pc=pc, N=N, dim=dim, Fd=Fd, Fs=Fs, base=base, u=_sparse_rows(N, Fs), top={})
    _cache[name] = c
    return c


def _order(c, combo, dense_mult, with_sparse):
    """Top-128 local rows and the int64 totals of one (pattern, sign) under a field composition (cached)."""
    key = (combo, dense_mult, with_sparse)
    if key not in c["top"]:
        T = dense_mult * X.dense_scores(*combo, c["N"])
        if with_sparse:
            T = T + c["u"].sum(axis=0)
        o = X.topk_order(T, 128)
        c["top"][key] = (o, T[o])
    return c["top"][key]


def _combos(Q, salt):
    return [X.COMBOS[(i * 7 + salt) % len(X.COMBOS)] for i in range(Q)]


def _queries(c, combos):
    return torch.from_numpy(np.stack([X.query_vector(p, s, c["dim"]) for p, s in combos])).to(DEV)


def _expected(c, combos, k, dense_mult, with_sparse, F, base):
    ids = np.empty((len(combos), k), dtype=np.int64)
    sc = np.empty((len(combos), k), dtype=np.float32)
    for i, cb in enumerate(combos):
        o, T = _order(c, cb, dense_mult, with_sparse)
        ids[i] = o[:k] + base
        sc[i] = (T[:k].astype(np.float64) / F).astype(np.float32)
    return torch.from_numpy(sc), torch.from_numpy(ids)


def _assert_exact(s, i, want_s, want_i, combos, what):
    s, i = s.cpu(), i.cpu()
    if torch.equal(i, want_i) and torch.equal(s, want_s):
        return
    bad = [q for q in range(want_i.shape[0]) if not (torch.equal(i[q], want_i[q]) and torch.equal(s[q], want_s[q]))]
    q = bad[0]
    j = int((i[q] != want_i[q]).nonzero()[0]) if not torch.equal(i[q], want_i[q]) else int((s[q] != want_s[q]).nonzero()[0])
    raise AssertionError(f"{what}: {len(bad)} of {want_i.shape[0]} queries wrong, first q={q} {combos[q]} rank {j}: "
                         f"got ({s[q, j].item()}, {i[q, j].item()}), want ({want_s[q, j].item()}, {want_i[q, j].item()})")


def _retriever(c, n_sparse=0, base=None, masked=None, top_k=100):
    from mfar_b200.modeling.retrieval import MultiFieldRetriever
    from mfar_b200.modeling.weighting import LinearWeights
    F = c["Fd"] + n_sparse
    layer = LinearWeights(F, 1).to(DEV)                # equal static logits: weights exactly 1/F
    r = MultiFieldRetriever(c["pc"], layer, n_sparse=n_sparse, top_k=top_k,
                            doc_id_base=c["base"] if base is None else base)
    if masked is not None:
        r.mask_field(masked)
    w = layer.field_weights(None, r.mask, batch=1)
    want = torch.full((1, F), 1.0 / F, device=DEV) * r.mask.reshape(1, F)
    assert torch.equal(w, want), "mixture weights are not exactly 1/F: the closed form does not apply"
    return r


def _sparse_tensor(c, Q, dtype=torch.float16, ld=None):
    N = c["N"]
    ld = ld or (N + 63) // 64 * 64
    sp = torch.zeros((Q, c["Fs"], ld), dtype=dtype, device=DEV)
    sp[:, :, :N] = torch.from_numpy(c["u"]).to(DEV, dtype).unsqueeze(0)
    return sp


def _launches(levels, extra=0):
    return 2 + 4 * levels + extra                     # (prefix levels) + scoring kernel + merge (+ sparse pre-mix)


# ---------------------------------------------------------------------------------------------- dense search
SMALL_RUNS = [(c, impl, Q) for c in ("s129", "s4097", "s4097_d64") for impl in IMPLS for Q in QS]


@pytest.mark.parametrize("corpus,impl,Q", SMALL_RUNS, ids=[f"{c}-{i}-Q{q}" for c, i, q in SMALL_RUNS])
def test_search_small_exact(corpus, impl, Q):
    c = _corpus(corpus)
    r = _retriever(c)
    combos = _combos(Q, salt=Q)
    q = _queries(c, combos)
    for k in KS:
        if k > c["N"]:
            continue
        s, i = r.search(q, top_k=k, impl=impl)
        assert r.last_launches == _launches(0)
        ws, wi = _expected(c, combos, k, c["Fd"], False, c["Fd"], c["base"])
        _assert_exact(s, i, ws, wi, combos, f"{corpus} {impl} Q={Q} k={k}")


# (impl, Q, {k: expected prefix levels}).  m330k: 2579 tiles, 2 dense fields; l4m: 31251 tiles, 1 field, ids up to 2^32-1
MID_RUNS = [("simt", 1, {1: 0, 100: 0, 128: 0}), ("simt", 17, {100: 0}),
            ("tcgen05", 17, {100: 0, 128: 0}), ("tcgen05", 32, {1: 1, 100: 1}), ("tcgen05", 65, {2: 1, 127: 1}),
            ("tcgen05", 129, {1: 1, 100: 2}), ("tcgen05_qs", 33, {100: 1}), ("tcgen05_qs", 129, {128: 1}),
            ("tcgen05_qs", 257, {2: 1, 100: 2}), ("auto", 64, {100: 1}), ("auto", 384, {1: 1, 128: 2}),
            ("auto", 512, {2: 1, 100: 2, 127: 2})]
LARGE_RUNS = [("simt", 1, {100: 0}), ("tcgen05", 1, {1: 0, 128: 0}), ("tcgen05_qs", 17, {100: 0}),
              ("tcgen05", 32, {1: 1, 100: 2}), ("tcgen05", 64, {2: 1, 128: 2}), ("tcgen05_qs", 64, {1: 1, 100: 2}),
              ("auto", 64, {127: 2}), ("auto", 129, {100: 2}), ("tcgen05", 512, {1: 2, 100: 2}),
              ("auto", 384, {1: 1, 100: 2})]      # auto Q=384 on one field: query-stationary with two epilogue sets
BIG = [("m330k",) + r for r in MID_RUNS] + [("l4m",) + r for r in LARGE_RUNS]


@pytest.mark.parametrize("corpus,impl,Q,levels", BIG, ids=[f"{c}-{i}-Q{q}" for c, i, q, _ in BIG])
def test_search_at_scale_exact(corpus, impl, Q, levels):
    c = _corpus(corpus)
    r = _retriever(c)
    combos = _combos(Q, salt=3 * Q + 1)
    q = _queries(c, combos)
    for k, lv in levels.items():
        s, i = r.search(q, top_k=k, impl=impl)
        assert r.last_launches == _launches(lv), f"k={k}: {r.last_launches} launches, want {lv} prefix levels"
        ws, wi = _expected(c, combos, k, c["Fd"], False, c["Fd"], c["base"])
        _assert_exact(s, i, ws, wi, combos, f"{corpus} {impl} Q={Q} k={k}")


# ---------------------------------------------------------------------------------------------- sparse layouts
SPARSE_RUNS = [(c, i, q, lay) for c, i, q in
               [("s4097", "tcgen05", Q) for Q in (1, 17, 64)] + [("s4097", "auto", Q) for Q in (65, 257, 512)] +
               [("s4097", "simt", 33), ("m330k", "tcgen05", 64), ("m330k", "auto", 512)]
               for lay in ("f16_aligned", "f16_unaligned", "f32", "coo")
               if not (lay == "coo" and c == "m330k" and q > 64)]   # COO pairs of 512 x 330k rows: covered at 4097 docs


@pytest.mark.parametrize("corpus,impl,Q,layout", SPARSE_RUNS, ids=[f"{c}-{i}-Q{q}-{l}" for c, i, q, l in SPARSE_RUNS])
def test_search_sparse_layouts_exact(corpus, impl, Q, layout):
    """Dense fields carry the pattern, two sparse fields add tied integers: (2 v + u0 + u1) / 4 is exact.  Aligned f16
    rows take the fused epilogue gather (tensor-core kernels), an unaligned pitch the pre-mix kernel, COO pairs the
    scatter; the seeded 330k cases start their main pass behind a scored prefix."""
    c = _corpus(corpus)
    base = 0 if layout == "coo" else c["base"]          # COO rows are int32 GLOBAL doc rows
    r = _retriever(c, n_sparse=c["Fs"], base=base)
    combos = _combos(Q, salt=5 * Q + 2)
    q = _queries(c, combos)
    N, F = c["N"], c["Fd"] + c["Fs"]
    kw = {}
    if layout == "coo":
        u = torch.from_numpy(c["u"]).to(DEV)
        keys, vals, off = [], [], [0]
        for j in range(c["Fs"]):
            nz = u[j].nonzero().flatten().int()
            qq = torch.arange(Q, device=DEV, dtype=torch.int32).repeat_interleave(nz.numel())
            keys.append(torch.stack([qq, nz.repeat(Q)], dim=1))
            vals.append(u[j][nz.long()].half().repeat(Q))
            off.append(off[-1] + Q * nz.numel())
        kw["sparse_coo"] = (torch.cat(keys).contiguous(), torch.cat(vals).contiguous(), off)
    else:
        dtype = torch.float32 if layout == "f32" else torch.float16
        ld = N + 3 if layout == "f16_unaligned" else None
        kw["sparse"] = _sparse_tensor(c, Q, dtype, ld)
    for k in (1, 100, 128):
        s, i = r.search(q, top_k=k, impl=impl, **kw)
        ws, wi = _expected(c, combos, k, c["Fd"], True, F, base)
        _assert_exact(s, i, ws, wi, combos, f"{corpus} {layout} {impl} Q={Q} k={k}")


# ---------------------------------------------------------------------------------------------- sparse-only rows
def _row_values(combo, N, f32):
    """Per-query sparse row of a sparse-only scorer: sign * v(n), with -0.0 stored next to +0.0 for zero_sign."""
    name, sign = combo
    if not f32 and name in ("n", "perm", "div37"):
        name = "mod127"                                 # values above 2048 are not exact in f16
    v = X.dense_scores(name, sign, N).astype(np.float32)
    if name == "zero_sign":
        v[np.arange(N) % 3 == 1] = -0.0
    return (name, sign), v


@pytest.mark.parametrize("N", [4097, 330_001])
@pytest.mark.parametrize("dtype", ["f16", "f32"])
@pytest.mark.parametrize("Q", [1, 17, 64, 257])
def test_sparse_only_rows_exact(N, dtype, Q):
    """The streaming row top-k (no dense field) with its threshold-seed kernel (N >= 4096): planted rows have fewer
    than k nonzeros, so the seed and the k-th key sit on a tie of zeros; -0.0 must rank as 0.0."""
    from mfar_b200.modeling.retrieval import MultiFieldRetriever
    from mfar_b200.modeling.weighting import LinearWeights
    base = TOP - N
    r = MultiFieldRetriever(None, LinearWeights(1, 1).to(DEV), n_sparse=1, top_k=100, n_docs=N, device=DEV,
                            doc_id_base=base)
    f32 = dtype == "f32"
    combos, rows = [], []
    for cb in _combos(Q, salt=Q + N):
        cb, v = _row_values(cb, N, f32)
        combos.append(cb)
        rows.append(v)
    tdt = torch.float32 if f32 else torch.float16
    sp = torch.from_numpy(np.stack(rows)).to(DEV, tdt).unsqueeze(1).contiguous()
    assert bool((torch.signbit(sp) & (sp == 0)).any()) == any(cb[0] == "zero_sign" for cb in combos)
    for k in KS:
        s, i = r.search(None, sparse=sp, top_k=k, batch=Q)
        assert r.last_launches == 4                    # pre-mix + threshold seed + row scan + merge
        ws = np.empty((Q, k), dtype=np.float32)
        wi = np.empty((Q, k), dtype=np.int64)
        for qi, cb in enumerate(combos):
            T = X.dense_scores(*cb, N)
            o = X.topk_order(T, k)
            ws[qi], wi[qi] = T[o], o + base
        _assert_exact(s, i, torch.from_numpy(ws), torch.from_numpy(wi), combos, f"rows N={N} {dtype} Q={Q} k={k}")


# ---------------------------------------------------------------------------------------------- other entry points
def test_search_host_exact():
    c = _corpus("s4097")
    r = _retriever(c, n_sparse=c["Fs"])
    for Q, impl in ((17, "tcgen05"), (129, "auto")):
        combos = _combos(Q, salt=11)
        q = r.corpus.prepare_queries(_queries(c, combos)).cpu().pin_memory()
        sp = _sparse_tensor(c, Q)[:, :, :c["N"]].cpu().contiguous()
        for k in (2, 128):
            s, i = r.search_host(q, None, sp, top_k=k, impl=impl)
            ws, wi = _expected(c, combos, k, c["Fd"], True, c["Fd"] + c["Fs"], c["base"])
            _assert_exact(s, i, ws, wi, combos, f"search_host Q={Q} k={k}")


def test_graphed_search_exact():
    from mfar_b200.modeling.retrieval import GraphedSearch
    c = _corpus("s4097")
    r = _retriever(c, n_sparse=c["Fs"])
    Q, k = 64, 100
    g = GraphedSearch(r, Q, sparse="dense", top_k=k)
    for salt in (0, 9):                                # two replays with different batches
        combos = _combos(Q, salt)
        s, i = g(_queries(c, combos), None, _sparse_tensor(c, Q))
        ws, wi = _expected(c, combos, k, c["Fd"], True, c["Fd"] + c["Fs"], c["base"])
        _assert_exact(s, i, ws, wi, combos, f"GraphedSearch salt={salt}")


def test_mask_sweep_exact():
    """Field 1 carries the REVERSED doc order of field 0's pattern, so a masked field that leaks changes the order."""
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    N, dim = 4097, 768
    base = TOP - N
    docs = torch.from_numpy(X.doc_matrix(N, dim)).to(DEV).to(torch.bfloat16)
    pc = PackedCorpus(N, 2, dim, DEV)
    pc.load_rows(0, 0, docs)
    pc.load_rows(1, 0, docs.flip(0).contiguous())
    r = MultiFieldRetriever(pc, LinearWeights(2, 1).to(DEV), top_k=100, doc_id_base=base)
    for Q in (17, 257):
        combos = _combos(Q, salt=Q)
        q = torch.from_numpy(np.stack([X.query_vector(p, s, dim) for p, s in combos])).to(DEV)
        sets = [[], [0], [1]]
        for k in (1, 100, 128):
            s, i = r.search_mask_sweep(q, sets, top_k=k)
            for m, masked in enumerate(sets):
                ws = np.empty((Q, k), dtype=np.float32)
                wi = np.empty((Q, k), dtype=np.int64)
                for qi, cb in enumerate(combos):
                    v = X.dense_scores(*cb, N)
                    T = (v if 0 not in masked else 0) + (v[::-1] if 1 not in masked else 0)
                    T = np.broadcast_to(T, (N,)).astype(np.int64)
                    o = X.topk_order(T, k)
                    ws[qi], wi[qi] = (T[o] / 2.0).astype(np.float32), o + base
                _assert_exact(s[m], i[m], torch.from_numpy(ws), torch.from_numpy(wi), combos,
                              f"mask sweep {masked} Q={Q} k={k}")


@pytest.mark.parametrize("corpus", ["s4097", "m330k"])
def test_per_field_topk_dense_exact(corpus):
    """``per_field_topk`` ranks each field alone (weight 1): dense field scores are the pattern's integers.  Without the
    (0.0, row 0) initialisation the rule is (score desc, row asc); with it, negative entries become (0.0, row 0)."""
    c = _corpus(corpus)
    r = _retriever(c, n_sparse=c["Fs"])
    Q = 40
    combos = _combos(Q, salt=13)
    q = _queries(c, combos)
    sp = _sparse_tensor(c, Q)
    for k in (2, 100, 128):
        for zero_init in (False, True):
            s, i = r.per_field_topk(q, sp, top_k=k, zero_init=zero_init)
            ws, wi = _expected(c, combos, k, 1, False, 1, 0)
            if zero_init:
                neg = ws < 0
                ws, wi = ws.masked_fill(neg, 0.0), wi.masked_fill(neg, 0)
            for f in range(c["Fd"]):
                _assert_exact(s[f], i[f], ws, wi, combos, f"per_field_topk field {f} k={k} zero_init={zero_init}")
            for j in range(c["Fs"]):                   # sparse fields: the same u_j row for every query
                o = X.topk_order(c["u"][j], k)
                want_s = torch.from_numpy(c["u"][j][o].astype(np.float32)).expand(Q, k)
                want_i = torch.from_numpy(o.astype(np.int64)).expand(Q, k)
                _assert_exact(s[c["Fd"] + j], i[c["Fd"] + j], want_s, want_i, combos, f"per_field_topk sparse {j}")


# ---------------------------------------------------------------------------------------------- shards and exchange
def _shard_keys(c, q, k, cuts, impl="auto"):
    from mfar_b200.modeling.retrieval import MultiFieldRetriever
    parts = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        sh = MultiFieldRetriever(c["pc"].window(lo, hi - lo), _retriever(c).mixture, top_k=k,
                                 doc_id_base=c["base"] + lo)
        parts.append(sh.search(q, top_k=k, return_keys=True, impl=impl)[2])
    return torch.stack(parts)


@pytest.mark.parametrize("Q", [17, 129])
def test_virtual_shards_merge_and_exchange_exact(Q):
    """Doc-range shards whose cuts fall inside tie groups (128128 is inside a div37 and a div1000 run), each scored with
    global ids, merged by ``dist.merge_keys`` and by the peer exchange with virtual ranks: both equal the closed form."""
    from mfar_b200.dist import PeerExchange, merge_keys
    c = _corpus("m330k")
    cuts = [0, 128 * 1001, 128 * 2002, c["N"]]
    combos = _combos(Q, salt=17)
    q = _queries(c, combos)
    R = len(cuts) - 1
    for k in (1, 100, 128):
        keys = _shard_keys(c, q, k, cuts)
        ws, wi = _expected(c, combos, k, c["Fd"], False, c["Fd"], c["base"])
        s, i = merge_keys(keys, k)
        _assert_exact(s, i, ws, wi, combos, f"merge_keys Q={Q} k={k}")
        if Q > 17:                                     # every rank's exchange CTAs must be co-resident on one device
            continue
        n = PeerExchange.buffer_bytes(R, 256, 128)
        bufs = [torch.zeros(n, dtype=torch.uint8, device=DEV) for _ in range(R)]
        ex = [PeerExchange(256, 128, peer_buffers=bufs, rank=rk, world=R) for rk in range(R)]
        streams = [torch.cuda.Stream() for _ in range(R)]
        torch.cuda.synchronize()
        outs = []
        for rk in range(R):
            with torch.cuda.stream(streams[rk]):
                outs.append(ex[rk].merge(keys[rk], k))
        torch.cuda.synchronize()
        for rk, (s_r, i_r) in enumerate(outs):
            _assert_exact(s_r, i_r, ws, wi, combos, f"PeerExchange rank {rk} Q={Q} k={k}")


# ---------------------------------------------------------------------------------------------- BM25 retrieve, k > 128
@pytest.mark.parametrize("k", [150, 300])
def test_bm25_retrieve_pass_boundary_inside_tie_group(k):
    """``retrieve`` above 128 takes the ranking in passes of <= 128 and sinks the taken docs to -inf.  Docs repeat in
    classes of ~67 identical token lists, so ranks 128 and 256 fall inside groups of bit-identical scores; the
    documented rule is (score desc, row asc)."""
    from mfar_b200.data.bm25 import DeviceBM25
    N, V = 2000, 12
    docs = [[i % 5] * (1 + (i // 5) % 2) + [5 + i % 3] for i in range(N)]
    bm = DeviceBM25(device=DEV).index(docs, vocab=V)
    queries = [[0], [5], [1, 6], [11], [0, 0]]            # single-token (or one repeated) queries: one add per doc
    rows, scores = bm.retrieve(queries, k=k)
    full = bm.get_scores_batch(queries).cpu().numpy()
    n = np.arange(N)
    for qi in range(len(queries)):
        o = np.lexsort((n, -full[qi].astype(np.float64)))[:k]
        tied = int((full[qi] == full[qi][o[127]]).sum())
        assert tied > 1 or qi == 2
        assert np.array_equal(rows[qi], o), f"query {queries[qi]}: rows differ at rank {int(np.argmax(rows[qi] != o))}"
        assert np.array_equal(scores[qi], full[qi][o])


# ---------------------------------------------------------------------------------------------- direct merge
def _merge_case(L, Q, k_in, seed, tie_frac, zero_frac):
    from mfar_b200.dist import encode_keys
    g = np.random.default_rng(seed)
    scores = np.where(g.random((L, Q, k_in)) < tie_frac, 5.0, g.integers(-50, 50, (L, Q, k_in))).astype(np.float32)
    ids = g.permutation(L * Q * k_in).reshape(L, Q, k_in).astype(np.int64) * 3 + 7   # ids out of order in each list
    keys = encode_keys(scores, ids)
    keys[g.random((L, Q, k_in)) < zero_frac] = 0                                      # empty slots mixed in
    return keys


@pytest.mark.parametrize("L,Q,k_in,tie_frac,zero_frac", [
    (12, 5, 128, 0.9, 0.1),      # > 1024 keys share the cut's score word: the streaming path
    (320, 3, 128, 0.5, 0.2),     # L * k_in = 40960 > 38912 (sc_cap): the streaming path from the first phase
    (320, 2, 128, 1.0, 0.0),     # every key ties, none empty
    (3, 4, 100, 0.0, 0.3),       # tie-free control, ~30 % empty slots
    (2, 3, 40, 0.5, 0.5),        # fewer than k keys: (-inf, -1) padding
])
def test_merge_keys_direct(L, Q, k_in, tie_frac, zero_frac):
    """``mfar_topk_merge`` through ``dist.merge_keys``: every non-empty key is a candidate; the answer is a numpy sort
    of the keys."""
    from mfar_b200.dist import decode_keys, merge_keys
    keys = _merge_case(L, Q, k_in, 1 + L + Q, tie_frac, zero_frac)
    dev = torch.from_numpy(keys.view(np.int64)).to(DEV)
    for k in (1, 100, 128):
        s, i = merge_keys(dev, k)
        srt = np.sort(keys.transpose(1, 0, 2).reshape(Q, -1), axis=1)[:, ::-1][:, :k]
        if srt.shape[1] < k:
            srt = np.pad(srt, ((0, 0), (0, k - srt.shape[1])))
        ws, wi = decode_keys(srt)
        assert torch.equal(i.cpu(), torch.from_numpy(wi.astype(np.int64))), f"L={L} Q={Q} k_in={k_in} k={k}: ids"
        assert torch.equal(s.cpu(), torch.from_numpy(ws)), f"L={L} Q={Q} k_in={k_in} k={k}: scores"


# ---------------------------------------------------------------------------------------------- premise on the GPU
def test_fp32_checker_agrees_with_closed_form():
    """tests/checker.py (plain torch fp32, TF32 off) reproduces the closed-form scores of the 330k corpus: the exactness
    premise holds on the GPU's own fp32 arithmetic.  (Its ids are not compared: its chunked torch.topk does not order
    ties.)"""
    from checker import Fp32Checker
    c = _corpus("m330k")
    r = _retriever(c)
    combos = _combos(40, salt=0)
    qb = r.corpus.prepare_queries(_queries(c, combos))
    w = torch.full((40, c["Fd"]), 1.0 / c["Fd"], device=DEV)
    s, _ = Fp32Checker(c["pc"], doc_id_base=c["base"]).topk(qb, w, 128, slack=0)
    ws, _ = _expected(c, combos, 128, c["Fd"], False, c["Fd"], c["base"])
    assert torch.equal(s.cpu(), ws)


def test_zz_release_hbm():
    _free()
