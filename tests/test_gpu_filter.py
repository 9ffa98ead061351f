"""Filtered search (DESIGN §4.5) on the GPU, compared element for element.

Every input is integer-exact (doc coordinates 0..15, query coefficients -15..15, mixture weights 1/F with F in {1, 2},
sparse scores small integers in f16), so every score is an exact fp32 number in any summation order, in bf16 and in
E4M3, and the answer is the (score desc, id asc) order of the ELIGIBLE docs (tests/filter_oracle.py) - no tolerance.
Covered: every impl and both corpus dtypes at Q = 1 .. 512, doc_id_base 0 / 37 / 2^32 - N - 5 with a ragged last tile,
every sparse layout, the sparse-only scorer (its seed kernel), the single-field pair path and the 4-CTA clusters, filters
that keep all / none / fewer than k docs, shared and per-query rows, ineligible NaN / inf docs, the best docs placed in
the threshold-seeding prefix and left out, shards at unaligned bases, graph replays, and at C4 / C5-shard size the
unfiltered ranks 65..128 recovered by leaving out ranks 1..64.
"""
import gc

import numpy as np
import pytest
import torch

import filter_oracle as FO
from mfar_b200.data.bm25 import safe_docs_bitmap

pytestmark = pytest.mark.gpu

DEV = "cuda"
D = 128
N = 5000                          # 40 tiles, the last one holds 8 docs
K = 100
TOP = 1 << 32
IMPLS = ("simt", "tcgen05", "tcgen05_qs", "auto")
QS = (1, 20, 64, 65, 130, 512)
_cache = {}


def _free():
    _cache.clear()
    gc.collect()
    torch.cuda.empty_cache()


def _retriever(pc, n_fields, Fs=0, doc_id_base=0, top_k=K, sparse_indices=None, n_docs=None):
    from mfar_b200.modeling.retrieval import MultiFieldRetriever
    from mfar_b200.modeling.weighting import LinearWeights
    layer = LinearWeights(n_fields, 1)                    # softmax of zeros: every weight is exactly 1/F
    with torch.no_grad():
        layer.weight.zero_()
    return MultiFieldRetriever(pc, layer.to(DEV), n_sparse=Fs, top_k=top_k, doc_id_base=doc_id_base,
                               sparse_indices=sparse_indices, n_docs=n_docs, device=DEV)


def _int_fields(n, Fd, seed, hi=16):
    rng = np.random.default_rng(seed)
    dup = rng.integers(0, hi, size=(61, D))
    out = []
    for _ in range(Fd):
        x = rng.integers(0, hi, size=(n, D))
        m = rng.random(n) < 0.3                           # exact duplicates: tie groups across tiles
        x[m] = dup[rng.integers(0, 61, size=int(m.sum()))]
        out.append(x.astype(np.float32))
    return out


def _int_queries(Q, seed, lo=-15):
    q = np.random.default_rng(seed).integers(lo, 16, size=(Q, D)).astype(np.float32)
    if lo < 0:
        q[0] = 0                                          # every doc ties
    return q


def _small(dtype, Fd=2):
    key = ("small", dtype, Fd)
    if key not in _cache:
        from mfar_b200.modeling.retrieval import PackedCorpus
        fields = _int_fields(N, Fd, 7 + Fd)
        pc = PackedCorpus.from_fields([torch.from_numpy(f) for f in fields], DEV, dtype=dtype)
        q = _int_queries(512, 11)
        dense = sum(f.astype(np.float64) @ q.astype(np.float64).T for f in fields).T       # [512, N]
        _cache[key] = dict(pc=pc, fields=fields, q=q, dense=dense)
    return _cache[key]


def _bits(el, base):
    """Device int32 bitmap over global ids: [W] for one bool row [N], [R, W] for [R, N] (safe_docs_bitmap rows)."""
    b = FO.bitmap_rows(el, base).view(np.int32)
    return torch.from_numpy(b[0] if np.ndim(el) == 1 else b).to(DEV)


def _eq(got, want, what):
    s, i = got[0].cpu(), got[1].cpu()
    ws, wi = torch.from_numpy(want[0]), torch.from_numpy(want[1])
    if torch.equal(i, wi) and torch.equal(s, ws):
        return
    bad = (i != wi).any(1) | (s != ws).any(1)
    q = int(bad.nonzero()[0])
    j = int(((i[q] != wi[q]) | (s[q] != ws[q])).nonzero()[0])
    raise AssertionError(f"{what}: {int(bad.sum())} of {i.shape[0]} queries wrong, first q={q} rank {j}: got "
                         f"({s[q, j].item()}, {i[q, j].item()}), want ({ws[q, j].item()}, {wi[q, j].item()})")


def _filters(Q, n, seed):
    """name -> bool eligibility [n] (shared) or [Q, n] (per query)."""
    rng = np.random.default_rng(seed)
    few = np.zeros(n, dtype=bool)
    few[rng.choice(n, 40, replace=False)] = True          # fewer than k eligible docs
    dens = rng.choice([0.01, 0.5, 0.99], size=(Q, 1))
    return {"ones": np.ones(n, dtype=bool), "zeros": np.zeros(n, dtype=bool), "few": few,
            "shared50": rng.random(n) < 0.5, "shared1": rng.random(n) < 0.01,
            "per_query": rng.random((Q, n)) < dens}


RUNS = [(impl, dt, Q, base) for impl in IMPLS for dt in ("bf16", "e4m3") for Q in QS for base in (0, 37)
        if not (impl == "tcgen05_qs" and dt == "e4m3")]


@pytest.mark.parametrize("impl,dtype,Q,base", RUNS, ids=[f"{i}-{d}-Q{q}-b{b}" for i, d, q, b in RUNS])
def test_filtered_search_exact(impl, dtype, Q, base):
    c = _small(dtype)
    r = _retriever(c["pc"], 2, doc_id_base=base)
    q = torch.from_numpy(c["q"][:Q]).to(DEV)
    scores = c["dense"][:Q] / 2
    s0, i0, k0 = r.search(q, impl=impl, return_keys=True)
    for name, el in _filters(Q, N, seed=Q + base).items():
        bits = _bits(el, base)
        s, i, keys = r.search(q, impl=impl, doc_filter=bits, return_keys=True)
        what = f"{impl} {dtype} Q={Q} base={base} filter={name}"
        _eq((s, i), FO.filtered_topk(scores, el, K, base), what)
        if name == "ones":                                # the unfiltered call, bit for bit, keys too
            assert torch.equal(s, s0) and torch.equal(i, i0) and torch.equal(keys, k0), what
        if name == "zeros":
            assert (i == -1).all() and torch.isneginf(s).all(), what


HIGH = [(impl, "bf16", Q) for impl in IMPLS for Q in (1, 20)] + [(impl, "e4m3", Q) for impl in ("simt", "tcgen05")
                                                                 for Q in (1, 20)]


@pytest.mark.parametrize("impl,dtype,Q", HIGH, ids=[f"{i}-{d}-Q{q}" for i, d, q in HIGH])
def test_filtered_search_at_the_top_of_the_id_range(impl, dtype, Q):
    """Ids up to 2^32 - 6: one shared row covers 2^32 bits (512 MB), its word offsets need 64 bits."""
    base = TOP - N - 5
    c = _small(dtype)
    r = _retriever(c["pc"], 2, doc_id_base=base)
    q = torch.from_numpy(c["q"][:Q]).to(DEV)
    rng = np.random.default_rng(99)
    for name, el in (("ones", np.ones(N, dtype=bool)), ("shared50", rng.random(N) < 0.5), ("few", rng.random(N) < 0.006)):
        if ("high", name) not in _cache:                  # three 512 MB rows, kept for every case of this test
            _cache[("high", name)] = torch.from_numpy(
                safe_docs_bitmap(np.flatnonzero(el) + base, base + N).view(np.int32)).to(DEV)
        got = r.search(q, impl=impl, doc_filter=_cache[("high", name)])
        _eq(got, FO.filtered_topk(c["dense"][:Q] / 2, el, K, base), f"{impl} {dtype} Q={Q} high base {name}")


def test_ineligible_nan_and_inf_docs_never_appear():
    from mfar_b200.modeling.retrieval import PackedCorpus
    fields = _int_fields(N, 2, 21)
    fields[0][10, 0] = np.inf
    fields[0][20, 3] = np.nan
    fields[1][N - 1, 5] = -np.inf
    fields[1][700, :] = np.inf
    pc = PackedCorpus.from_fields([torch.from_numpy(f) for f in fields], DEV)
    r = _retriever(pc, 2, doc_id_base=37)
    rng = np.random.default_rng(5)
    for Q in (1, 20, 130):
        qn = _int_queries(Q, 22)
        qn[:, 0] = np.where(np.arange(Q) % 2 == 0, 3.0, -3.0)
        q = torch.from_numpy(qn).to(DEV)
        with np.errstate(invalid="ignore"):
            scores = sum(f.astype(np.float64) @ qn.astype(np.float64).T for f in fields).T / 2
        el = rng.random((Q, N)) < 0.5
        el[:, [10, 20, 700, N - 1]] = False
        for impl in IMPLS:
            s, i = r.search(q, impl=impl, doc_filter=_bits(el, 37))
            assert torch.isfinite(s[i >= 0]).all(), impl
            _eq((s, i), FO.filtered_topk(scores, el, K, 37), f"{impl} Q={Q} nonfinite ineligible")


# ---------------------------------------------------------------------------------------------- sparse inputs
LAYOUTS = [(lay, impl, dt) for lay in ("rows_f16", "rows_f32_unaligned", "coo", "bm25")
           for impl in ("simt", "tcgen05", "tcgen05_qs") for dt in ("bf16", "e4m3")
           if not (impl == "tcgen05_qs" and dt == "e4m3")]


def _bm25(n, V=300, seed=31):
    from mfar_b200.data.bm25 import DeviceBM25
    rng = np.random.default_rng(seed)
    docs = [rng.integers(0, V, size=rng.integers(1, 12)).tolist() for _ in range(n)]
    return DeviceBM25(device=DEV).index(docs, vocab=V)


@pytest.mark.parametrize("layout,impl,dtype", LAYOUTS, ids=[f"{a}-{b}-{c}" for a, b, c in LAYOUTS])
def test_sparse_layouts_exact(layout, impl, dtype):
    c = _small(dtype, Fd=1)
    base, Q = 37, 65
    rng = np.random.default_rng(3)
    qn = c["q"][:Q]
    q = torch.from_numpy(qn).to(DEV)
    el = rng.random((Q, N)) < rng.choice([0.02, 0.5], size=(Q, 1))
    bits = _bits(el, base)
    kw = {}
    if layout == "bm25":
        idx = _bm25(N)
        r = _retriever(c["pc"], 2, Fs=1, doc_id_base=base, sparse_indices=[idx])
        tokens = [[[int(t)] for t in rng.integers(0, 300, size=Q)]]      # one token: one exact add per doc
        sp = r.bm25_field_scores(tokens, Q)[:, 0, :N].double().cpu().numpy()
        kw["sparse_tokens"] = tokens
    else:
        r = _retriever(c["pc"], 2, Fs=1, doc_id_base=base)
        u = (rng.integers(0, 16, size=(Q, N)) * (rng.random((Q, N)) < 0.4)).astype(np.float64)
        sp = u
        if layout == "coo":
            qq, dd = np.nonzero(u)
            keys = torch.from_numpy(np.stack([qq, dd + base], 1).astype(np.int32)).to(DEV)
            kw["sparse_coo"] = (keys, torch.from_numpy(u[qq, dd]).half().to(DEV), [0, len(qq)])
        else:
            f32 = layout == "rows_f32_unaligned"
            ld = N + 3 if f32 else (N + 63) // 64 * 64
            t = torch.zeros((Q, 1, ld), dtype=torch.float32 if f32 else torch.float16, device=DEV)
            t[:, 0, :N] = torch.from_numpy(u).to(DEV, t.dtype)
            kw["sparse"] = t
    scores = (c["dense"][:Q] + sp) / 2
    got = r.search(q, impl=impl, doc_filter=bits, **kw)
    _eq(got, FO.filtered_topk(scores, el, K, base), f"{layout} {impl} {dtype}")
    one = r.search(q, impl=impl, doc_filter=_bits(np.ones(N, dtype=bool), base), **kw)
    zero = r.search(q, impl=impl, **kw)
    if layout != "bm25":                                  # BM25: the fp32 atomics of the scatter may reorder
        assert torch.equal(one[0], zero[0]) and torch.equal(one[1], zero[1])


@pytest.mark.parametrize("Q", (1, 7, 64))
def test_sparse_only_scorer_and_its_seed_kernel(Q):
    """No dense field: the row top-k and its threshold seed (n_docs >= 4096; the seed scans the first 32768 docs).  The
    best scores sit in that prefix and are ineligible: a seed taken over them admits no eligible doc."""
    n, base = 40_000, 37
    rng = np.random.default_rng(Q)
    u = rng.integers(0, 2000, size=(Q, n)).astype(np.float64)
    poison = rng.choice(32768, 300, replace=False)
    u[:, poison] = 1e6 + rng.integers(0, 50, size=(Q, 300))
    sp = torch.from_numpy(u).float().to(DEV).unsqueeze(1).contiguous()
    r = _retriever(None, 1, Fs=1, doc_id_base=base, n_docs=n)
    el = rng.random((Q, n)) < 0.6
    el[:, poison] = False
    for rows in ("per_query", "shared"):
        e = el if rows == "per_query" else el[0]
        got = r.search(None, sparse=sp, doc_filter=_bits(e, base))
        _eq(got, FO.filtered_topk(u, e, K, base), f"sparse-only Q={Q} {rows}")


@pytest.mark.parametrize("Q", (130, 512))
def test_single_field_pair_path_and_4cta_clusters(Q):
    """One dense field at Q > 128: CTA pairs with two epilogue sets (ES = 2, alternate half-tiles); at Q = 512 the
    pairs of a worker column run as 4-CTA clusters."""
    from mfar_b200 import _native as nv
    c = _small("bf16", Fd=1)
    r = _retriever(c["pc"], 1, doc_id_base=37)
    q = torch.from_numpy(c["q"][:Q]).to(DEV)
    fl = _filters(Q, N, seed=Q)
    for name in ("per_query", "shared50", "few"):
        nv.lib().mfar_profile_cluster4_ctas()
        got = r.search(q, impl="tcgen05_qs", doc_filter=_bits(fl[name], 37))
        torch.cuda.synchronize()
        if Q == 512:
            assert nv.lib().mfar_profile_cluster4_ctas() > 0
        _eq(got, FO.filtered_topk(c["dense"][:Q], fl[name], K, 37), f"pair path Q={Q} {name}")


# ---------------------------------------------------------------------------------------------- poisoned prefix
def _device_filtered_topk(fields_t, q, el_t, k, base, F):
    """The filtered top-k of exact integer scores on the device, for shapes the host helper is too slow for: one int64
    key per doc, (2F * score) << 32 | (2^32 - 1 - global id), ineligible docs at the bottom."""
    s = sum(x.double() @ q.double().t() for x in fields_t).t()                       # [Q, n], exact integers
    ids = torch.arange(s.shape[1], device=DEV, dtype=torch.int64) + base
    key = (s.round().long() << 32) | (0xFFFFFFFF - ids)
    key = torch.where(el_t, key, torch.full_like(key, -(1 << 62)))
    top = key.topk(k, dim=1).values
    live = top != -(1 << 62)
    out_i = torch.where(live, 0xFFFFFFFF - (top & 0xFFFFFFFF), torch.full_like(top, -1))
    out_s = torch.where(live, (top >> 32).double() / F, torch.full_like(top, float("-inf"), dtype=torch.float64))
    return out_s.float().cpu().numpy(), out_i.cpu().numpy()


# (impl, Q, dense fields, prefix docs poisoned, prefix levels the call must run)
PREFIX = [("tcgen05", 64, 1, 148 * 128, 1), ("tcgen05", 512, 2, 18 * 32 * 128, 2), ("tcgen05_qs", 512, 2, 37 * 17 * 128, 2),
          ("auto", 512, 2, 37 * 17 * 128, 2)]


@pytest.mark.parametrize("impl,Q,Fd,P,levels", PREFIX, ids=[f"{p[0]}-Q{p[1]}-L{p[4]}" for p in PREFIX])
def test_best_docs_in_the_seeding_prefix_are_ineligible(impl, Q, Fd, P, levels):
    """The threshold-seeding prefix (csrc/capi.cu: 4 more launches per level) holds every query's best docs, all
    ineligible.  A prefix pass that ignored the filter would seed a threshold no eligible doc reaches."""
    from mfar_b200.modeling.retrieval import PackedCorpus
    n, base = 330_001, 37
    key = ("prefix", Fd, P, Q)
    if key not in _cache:
        _free()
        rng = np.random.default_rng(40 + Fd)
        fields = []
        for _ in range(Fd):
            x = rng.integers(0, 8, size=(n, D)).astype(np.float32)
            x[:P] = 15                                    # every query's best docs (query coefficients are positive)
            fields.append(x)
        pc = PackedCorpus.from_fields([torch.from_numpy(f) for f in fields], DEV)
        el = torch.from_numpy(rng.random((Q, n)) < 0.7)
        el[:, :P] = False
        el[:, :P:997] = True                              # a few prefix docs stay eligible
        bits = torch.from_numpy(FO.bitmap_rows(el.numpy(), base).view(np.int32)).to(DEV)
        _cache[key] = dict(pc=pc, fields=[torch.from_numpy(f).to(DEV) for f in fields], el=el.to(DEV), bits=bits)
    c = _cache[key]
    r = _retriever(c["pc"], Fd, doc_id_base=base)
    qn = _int_queries(Q, 43, lo=1)
    q = torch.from_numpy(qn).to(DEV)
    el, bits = c["el"][:Q], c["bits"][:Q]
    for rows in ("per_query", "shared"):
        b, e = (bits, el) if rows == "per_query" else (bits[0].contiguous(), el[:1].expand(Q, n))
        got = r.search(q, impl=impl, doc_filter=b)
        assert r.last_launches == 2 + 4 * levels, (r.last_launches, levels)
        _eq(got, _device_filtered_topk(c["fields"], q, e, K, base, Fd), f"{impl} Q={Q} prefix {rows}")


# ---------------------------------------------------------------------------------------------- shards and graphs
def test_shards_at_unaligned_bases_merge_to_the_unsharded_filtered_search():
    from mfar_b200.dist import ShardedRetriever, merge_keys
    from mfar_b200.modeling.retrieval import MultiFieldRetriever
    c = _small("bf16")
    base = 37
    r = _retriever(c["pc"], 2, doc_id_base=base)
    for Q, impl in ((1, "simt"), (20, "tcgen05"), (130, "tcgen05_qs"), (64, "auto")):
        q = torch.from_numpy(c["q"][:Q]).to(DEV)
        el = np.random.default_rng(Q).random((Q, N)) < 0.3
        bits = _bits(el, base)
        s, i, keys = r.search(q, impl=impl, doc_filter=bits, return_keys=True)
        _eq((s, i), FO.filtered_topk(c["dense"][:Q] / 2, el, K, base), f"unsharded Q={Q}")
        parts = []
        for lo, hi in ((0, 128 * 9), (128 * 9, 128 * 30), (128 * 30, N)):
            sh = MultiFieldRetriever(c["pc"].window(lo, hi - lo), r.mixture, top_k=K, doc_id_base=base + lo)
            k = min(K, hi - lo)
            ss, si, sk = sh.search(q, impl=impl, doc_filter=bits, top_k=k, return_keys=True)
            ws, wi = ShardedRetriever(sh).search(q, top_k=k, doc_filter=bits)         # one rank: the local merge
            assert torch.equal(ws, ss) and torch.equal(wi, si)
            parts.append(torch.nn.functional.pad(sk, (0, K - k)))
        ms, mi = merge_keys(torch.stack(parts), K)
        assert torch.equal(ms, s) and torch.equal(mi, i), f"merged shards Q={Q}"


@pytest.mark.parametrize("Q", (20, 130))
def test_graph_replays_read_the_filter_contents_at_replay_time(Q):
    from mfar_b200.modeling.retrieval import GraphedSearch
    c = _small("bf16")
    r = _retriever(c["pc"], 2, doc_id_base=37)
    q = torch.from_numpy(c["q"][:Q]).to(DEV)
    rng = np.random.default_rng(Q)
    bits = _bits(rng.random((Q, N)) < 0.5, 37)
    g = GraphedSearch(r, Q, doc_filter=bits)
    for step in range(3):
        el = rng.random((Q, N)) < (0.5, 0.02, 0.9)[step]
        bits.copy_(_bits(el, 37))
        gs, gi = g(q)
        es, ei = r.search(q, doc_filter=bits)
        assert torch.equal(gs, es) and torch.equal(gi, ei), step
        _eq((gs, gi), FO.filtered_topk(c["dense"][:Q] / 2, el, K, 37), f"graph step {step}")


# ---------------------------------------------------------------------------------------------- at scale
# name: (n_docs, dense fields, sparse fields, doc_id_base, seed)
SCALE = {"c4_amazon_hybrid": (957_192, 8, 8, 0, 103), "c5_shard_of_8": (1_250_000, 8, 0, 3_750_000, 104)}
SCALE_RUNS = [(c, Q, impl) for c in SCALE for Q in (64, 512) for impl in ("tcgen05", "tcgen05_qs", "auto")]


def _scale_case(name):
    if name in _cache:
        return _cache[name]
    _free()
    from mfar_b200 import synth as S
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    n, Fd, Fs, base, seed = SCALE[name]
    Dm = 768
    pc = PackedCorpus(n, Fd, Dm, DEV)
    S.fill_packed_corpus(pc, seed=seed)
    q = S.make_queries(512, Dm, S.corpus_mean(Dm, seed, DEV), seed + 1, DEV)
    layer = LinearWeights(Dm, Fd + Fs, query_cond=True)
    with torch.no_grad():
        layer.weight.copy_(S.make_mixture(Dm, Fd + Fs, seed + 2))
    sp = None
    if Fs:
        sp = torch.zeros((512, Fs, (n + 63) // 64 * 64), dtype=torch.float16, device=DEV)
        for q0 in range(0, 512, 32):
            sp[q0:q0 + 32, :, :n] = S.make_sparse(32, Fs, n, seed + 3 + q0, DEV)
    r = MultiFieldRetriever(pc, layer.to(DEV), n_sparse=Fs, top_k=128, doc_id_base=base)
    full = safe_docs_bitmap(np.arange(base, base + n), base + n)
    _cache[name] = dict(r=r, q=q, sp=sp, full=full, base=base)
    return _cache[name]


@pytest.mark.parametrize("case,Q,impl", SCALE_RUNS, ids=[f"{c}-Q{q}-{i}" for c, q, i in SCALE_RUNS])
def test_leaving_out_the_top_64_gives_ranks_65_to_128(case, Q, impl):
    """No oracle needed: with each query's unfiltered top 64 ineligible, the filtered top 64 is the unfiltered
    ranks 65..128, key for key (the same kernels score every doc the same way with and without a filter)."""
    c = _scale_case(case)
    r, q, sp = c["r"], c["q"][:Q], None if c["sp"] is None else c["sp"][:Q]
    _, i128, k128 = r.search(q, sparse=sp, top_k=128, impl=impl, return_keys=True)
    ids = i128[:, :64].cpu().numpy()
    rows = np.tile(c["full"], (Q, 1))
    np.bitwise_and.at(rows, (np.repeat(np.arange(Q), 64), (ids >> 5).ravel()),
                      ~(np.uint32(1) << (ids & 31).astype(np.uint32)).ravel())
    bits = torch.from_numpy(rows.view(np.int32)).to(DEV)
    _, i64, k64 = r.search(q, sparse=sp, top_k=64, impl=impl, return_keys=True, doc_filter=bits)
    assert torch.equal(k64, k128[:, 64:]), f"{case} Q={Q} {impl}"
    assert torch.equal(i64, i128[:, 64:])


def test_zz_release_hbm():
    _free()
