"""Cosine scoring (``PackedCorpus(normalize=True)``) against the float64 contract of ``mfar_oracle.normalize_rows_bf16``.

The scoring kernels do not see the flag: a cosine corpus is a corpus of unit rows.  So the tests pin the two places
where the flag acts - the pack kernel (docs) and ``prepare_queries`` (queries), bit for bit - and then every search
entry point on inputs whose cosine scores are exact.  A doc row holds +-c on an aligned block of 4^m coordinates, with c
of at most 8 significant bits anywhere from 2^-36 to 2^70: its unit row is exactly +-2^-m whatever c is, so every
cosine is a signed overlap count times a power of two, exact in fp32 in any summation order.  The magnitudes c grow
with the doc id, so the raw-dot top-k of a query shares almost nothing with its cosine top-k (asserted): a path that
skips or mangles the normalisation changes the answer, and the answer is compared with ``torch.equal``.
"""
import gc
import io

import numpy as np
import pytest
import torch

import exact_topk as X
import mfar_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda"
TOP = 2 ** 32
IMPLS = ("simt", "tcgen05", "tcgen05_qs", "auto")
EPS = float(np.float32(1e-12))


def _mods():
    from mfar_b200.modeling.retrieval import GraphedSearch, MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    return GraphedSearch, MultiFieldRetriever, PackedCorpus, LinearWeights


def _bits(x):
    """int16 bit patterns of bf16 values (float32 array / tensor holding bf16 values, or a bf16 tensor)."""
    if not torch.is_tensor(x):
        x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    return x.cpu().to(torch.bfloat16).view(torch.int16)


def _assert_bits(got, want, what):
    got, want = _bits(got), _bits(want)
    bad = got != want
    if bad.any():
        r, c = (int(v) for v in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements in {int(bad.any(1).sum())} rows "
                             f"differ; first at [{r},{c}]: got bits {int(got[r, c]) & 0xFFFF:#06x}, "
                             f"want {int(want[r, c]) & 0xFFFF:#06x}")


# ---------------------------------------------------------------------------------------------- 1. pack bit-exactness
def _edge_rows(dim):
    """Rows where a normalisation goes wrong: zero (with -0.0), one nonzero, norms either side of eps, fp32 subnormals,
    |x| >= 2^64 (fp32 squares overflow), the fp32 extremes, and signed zeros next to nonzeros."""
    z = np.zeros(dim, dtype=np.float32)
    rows = []
    rows.append(z.copy())
    r = z.copy(); r[1::2] = -0.0; rows.append(r)
    r = z.copy(); r[dim - 1] = -3.5; rows.append(r)
    r = z.copy(); r[0] = 2.0 ** 100; rows.append(r)
    r = z.copy(); r[:4] = EPS / 4; rows.append(r)                       # norm eps / 2: divided by eps
    r = z.copy(); r[:4] = EPS; rows.append(r)                           # norm 2 eps
    r = z.copy(); r[0], r[1] = 3 * 2.0 ** -43, 4 * 2.0 ** -43; rows.append(r)   # norm 5 * 2^-43 < eps
    r = z.copy(); r[::3] = 2.0 ** -140; r[1] = 3 * 2.0 ** -149; rows.append(r)  # fp32 subnormals only
    r = z.copy(); r[0] = 1.0; r[1::5] = 2.0 ** -135; rows.append(r)      # subnormal quotients
    r = (2.0 ** 64 * (1 + (np.arange(dim) % 7) / 8)).astype(np.float32); rows.append(r)
    r = z.copy(); r[0], r[dim // 2] = 1.8e19, -3e38; rows.append(r)
    r = z.copy(); r[::2] = -0.0; r[1] = 5.0; rows.append(r)
    r = np.full(dim, -7.0, dtype=np.float32); r[::4] = 7.0; rows.append(r)
    return np.stack(rows)


def _pack_rows(N, dim, seed):
    g = np.random.default_rng(seed)
    mu = g.standard_normal(dim)
    x = (g.standard_normal((N, dim)) + 0.5 * mu) * np.exp2(g.uniform(-70, 70, (N, 1)))
    x = x.astype(np.float32)
    e = _edge_rows(dim)
    if N >= 2 * len(e):
        x[:len(e)] = e
        x[N - len(e):] = e[::-1]
    return x


def _packed_field(pc, f, N):
    from mfar_b200.modeling.retrieval import TILE_DOCS
    tiles = pc.data.numel() // (pc.n_fields * TILE_DOCS * pc.dim_pad)
    return pc.data.view(tiles, pc.n_fields, TILE_DOCS, pc.dim_pad)[:, f].reshape(-1, pc.dim_pad)[:N]


@pytest.mark.parametrize("N", [1, 127, 129, 4097])
@pytest.mark.parametrize("dim", [32, 64, 100, 768, 1000, 1024])
@pytest.mark.parametrize("src", ["f32", "bf16"])
def test_pack_bit_exact(src, dim, N):
    """Packed bits of field 1 of 2, loaded in chunks of 77 rows (row_begin off the 128-doc tiles), equal the contract;
    padding columns are +0; a window of the corpus sees the same bits."""
    _, _, PackedCorpus, _ = _mods()
    x = torch.from_numpy(_pack_rows(N, dim, seed=dim * 7 + N))
    if src == "bf16":
        x = x.to(torch.bfloat16)
    want = O.normalize_rows_bf16(x)
    pc = PackedCorpus(N, 2, dim, DEV, normalize=True)
    pc.load_field(1, x.numpy() if src == "f32" else x, chunk_rows=77)     # a host array, as from a memmap
    got = _packed_field(pc, 1, N)
    _assert_bits(got[:, :dim], want, f"pack {src} dim={dim} N={N}")
    assert not _bits(got[:, dim:]).any(), "padding columns must be +0"
    assert not _bits(_packed_field(pc, 0, N)).any(), "field 0 was never loaded"
    if N > 128:
        w = pc.window(128, N - 128)
        _assert_bits(_packed_field(w, 1, N - 128)[:, :dim], want[128:], "window(128)")


@pytest.mark.parametrize("dim", [64, 100, 768])
@pytest.mark.parametrize("dtype", ["f32", "bf16", "f16"])
def test_prepare_queries_bit_exact(dtype, dim):
    """Queries get the treatment docs get: the same contract, from host or device, fp32 / bf16 / f16."""
    _, _, PackedCorpus, _ = _mods()
    tdt = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}[dtype]
    if dtype == "f16":                                   # f16 range: magnitudes 2^-8 .. 2^8, f16 subnormals, zeros
        g = np.random.default_rng(dim)
        x = (g.standard_normal((300, dim)) * np.exp2(g.uniform(-8, 8, (300, 1)))).astype(np.float32)
        x[0] = 0.0
        x[1] = -0.0
        x[2, 1:] = 0.0
        x[3, ::2] = 2.0 ** -20
        x[4, 1::2] = -0.0
    else:
        x = _pack_rows(300, dim, seed=11 + dim)
    q = torch.from_numpy(x).to(tdt)
    want = O.normalize_rows_bf16(q)
    pc = PackedCorpus(129, 1, dim, DEV, normalize=True)
    for where in ("host", "device"):
        got = pc.prepare_queries(q if where == "host" else q.to(DEV))
        assert got.dtype == torch.bfloat16 and got.is_cuda and got.is_contiguous() and got.shape == (300, pc.dim_pad)
        _assert_bits(got[:, :dim], want, f"prepare_queries {dtype} {where} dim={dim}")
        assert not _bits(got[:, dim:]).any()


def test_pack_and_queries_without_normalize_are_plain_bf16():
    """normalize=False is a plain round to bf16 of docs and queries (the raw-dot path must not change)."""
    _, _, PackedCorpus, _ = _mods()
    x = torch.from_numpy(_pack_rows(300, 100, seed=3))
    pc = PackedCorpus(300, 1, 100, DEV)
    pc.load_field(0, x, chunk_rows=77)
    _assert_bits(_packed_field(pc, 0, 300)[:, :100], x.to(torch.bfloat16).float(), "pack raw")
    _assert_bits(pc.prepare_queries(x)[:, :100], x.to(torch.bfloat16).float(), "queries raw")


# ---------------------------------------------------------------------------------------------- exact cosine inputs
def _levels(dim):
    return 3 if dim == 64 else 4                        # block sizes 4^0 .. 4^M fit the row


def _layout(N, dim):
    """Per doc: block level m, block index, sign and magnitude c (8 significant bits, 2^-36 <= c < 2^70).  c grows with
    the block size and, inside a level, with the id, so the raw dot prefers wide blocks and high ids where the cosine
    prefers the query's own level and low ids.  One doc in 61 is negative."""
    n = np.arange(N, dtype=np.int64)
    M = _levels(dim)
    m = n % (M + 1)
    blk = (n // 7) % (dim // 4 ** m)
    sign = np.where(n % 61 == 3, -1, 1)
    c = (128 + n % 128) * np.exp2(-43 + (84 // M) * m + (22 * n) // N)
    return m, blk, sign, c


def _doc_rows(lay, dim, lo, hi):
    m, blk, sign, c = (a[lo:hi] for a in lay)
    x = np.zeros((hi - lo, dim), dtype=np.float32)
    for lv in np.unique(m):
        rows = np.nonzero(m == lv)[0]
        size = 4 ** int(lv)
        cols = blk[rows, None] * size + np.arange(size)
        x[rows[:, None], cols] = (sign[rows] * c[rows])[:, None]
    return x


def _qspecs(Q, dim, salt):
    """(m, block, sign, c) per query; a quarter of them negative, c spans 2^-36 .. 2^70."""
    out = []
    for i in range(Q):
        j = i + salt
        mq = j % (_levels(dim) + 1)
        out.append((mq, (j * 5 + salt) % (dim // 4 ** mq), -1 if (j // 4) % 4 == 3 else 1,
                    float((128 + (37 * j) % 128) * 2.0 ** (-43 + (j * 13) % 106))))
    return out


def _query_rows(specs, dim):
    x = np.zeros((len(specs), dim), dtype=np.float32)
    for i, (mq, bq, sq, cq) in enumerate(specs):
        size = 4 ** mq
        x[i, bq * size:(bq + 1) * size] = sq * cq
    return x


def _cos_int(spec, lay):
    """int64 [N]: 256 * cosine of every doc (an integer: overlap 4^min(m, mq) times 2^-(m + mq))."""
    mq, bq, sq, _ = spec
    m, blk, sign, _ = lay
    big = 4 ** np.maximum(m, mq)
    nest = (blk * 4 ** m) // big == (bq * 4 ** mq) // big
    return np.where(nest, sq * sign * (256 >> np.abs(m - mq)), 0).astype(np.int64)


def _raw_dot(spec, lay):
    mq, bq, sq, cq = spec
    m, blk, sign, c = lay
    big = 4 ** np.maximum(m, mq)
    nest = (blk * 4 ** m) // big == (bq * 4 ** mq) // big
    return np.where(nest, sq * sign * cq * c * 4.0 ** np.minimum(m, mq), 0.0)


def _sparse_int(N, Fs):
    """int64 [Fs, N]: sparse scores in units of 2^-8 (exact in f16), the same for every query."""
    n = np.arange(N, dtype=np.int64)
    return np.stack([4 * ((n // 3) % 5), np.where(n % 7 == 2, 16, 0)])[:Fs]


_cache = {}


def _free():
    _cache.clear()
    gc.collect()
    torch.cuda.empty_cache()


def _corpus(name):
    """name: (N, dim, dense fields, sparse fields, chunk_rows)."""
    if name in _cache:
        return _cache[name]
    if name == "l4m":
        _free()
    _, _, PackedCorpus, _ = _mods()
    N, dim, Fd, Fs, chunk = {"s64": (4097, 64, 2, 2, 77), "s768": (4097, 768, 2, 2, 1000),
                             "l4m": (4_000_001, 64, 1, 0, None)}[name]
    lay = _layout(N, dim)
    pc = PackedCorpus(N, Fd, dim, DEV, normalize=True)
    src = np.empty((N, dim), dtype=np.float32)
    for lo in range(0, N, 1 << 18):
        src[lo:lo + (1 << 18)] = _doc_rows(lay, dim, lo, min(N, lo + (1 << 18)))
    for f in range(Fd):                                  # identical fields: fp32 memmap-like source, then bf16
        v = src if f == 0 else torch.from_numpy(src).to(torch.bfloat16)
        if chunk:
            pc.load_field(f, v, chunk_rows=chunk)
        else:
            pc.load_field(f, v)
    del src
    c = dict(pc=pc, N=N, dim=dim, Fd=Fd, Fs=Fs, lay=lay, base=TOP - N, u=_sparse_int(N, Fs), keys={})
    _cache[name] = c
    return c


def _key(c, spec, dense_mult, sparse_js):
    """int64 [N] totals in units of 2^-8 of one query under a field composition (cached by what it depends on)."""
    k = (spec[:3], dense_mult, tuple(sparse_js))
    if k in c["keys"]:
        return c["keys"][k]
    T = dense_mult * _cos_int(spec, c["lay"])
    for j in sparse_js:
        T = T + c["u"][j]
    if c["N"] < 100_000:                                # the 4M-doc totals are not kept
        c["keys"][k] = T
    return T


def _expected(c, specs, k, dense_mult, sparse_js, F, base):
    ids = np.empty((len(specs), k), dtype=np.int64)
    sc = np.empty((len(specs), k), dtype=np.float32)
    seen = {}
    for i, sp in enumerate(specs):
        if sp[:3] not in seen:                          # the cosine does not depend on the query's magnitude
            T = _key(c, sp, dense_mult, sparse_js)
            o = X.topk_order(T, k)
            seen[sp[:3]] = (o + base, (T[o].astype(np.float64) / (256.0 * F)).astype(np.float32))
        ids[i], sc[i] = seen[sp[:3]]
    return torch.from_numpy(sc), torch.from_numpy(ids)


def _assert_exact(s, i, want_s, want_i, what):
    s, i = s.cpu(), i.cpu()
    if torch.equal(i, want_i) and torch.equal(s, want_s):
        return
    bad = [q for q in range(want_i.shape[0]) if not (torch.equal(i[q], want_i[q]) and torch.equal(s[q], want_s[q]))]
    q = bad[0]
    j = int(((i[q] != want_i[q]) | (s[q] != want_s[q])).nonzero()[0])
    raise AssertionError(f"{what}: {len(bad)} of {want_i.shape[0]} queries wrong, first q={q} rank {j}: "
                         f"got ({s[q, j].item()}, {i[q, j].item()}), want ({want_s[q, j].item()}, {want_i[q, j].item()})")


def _retriever(c, n_sparse=0, base=None, top_k=100, pc=None):
    _, MultiFieldRetriever, _, LinearWeights = _mods()
    F = c["Fd"] + n_sparse
    layer = LinearWeights(F, 1).to(DEV)                 # equal static logits: weights exactly 1/F
    assert torch.equal(layer.field_weights(None, None, batch=1), torch.full((1, F), 1.0 / F, device=DEV))
    return MultiFieldRetriever(pc or c["pc"], layer, n_sparse=n_sparse, top_k=top_k,
                               doc_id_base=c["base"] if base is None else base)


def _sparse_tensor(c, Q, N=None):
    N = N or c["N"]
    ld = (N + 63) // 64 * 64
    sp = torch.zeros((Q, c["Fs"], ld), dtype=torch.float16, device=DEV)
    sp[:, :, :N] = (torch.from_numpy(c["u"][:, :N]).to(DEV, torch.float32) / 256).half().unsqueeze(0)
    return sp


# ---------------------------------------------------------------------------------------------- 2. exact cosine top-k
def test_raw_dot_would_rank_differently():
    """The premise: on these inputs the raw-dot top-k of a positive query shares at most 10 % of its ids with the
    cosine top-k, so a path that skips the normalisation cannot pass."""
    for name in ("s64", "s768"):
        N, dim = 4097, 64 if name == "s64" else 768
        lay = _layout(N, dim)
        for spec in _qspecs(64, dim, salt=1):
            if spec[2] < 0:
                continue
            for k in (100, 128):
                cos = set(X.topk_order(_cos_int(spec, lay), k).tolist())
                raw = _raw_dot(spec, lay)
                rawk = set(np.lexsort((np.arange(N), -raw))[:k].tolist())
                assert len(cos & rawk) <= k // 10, f"{name} {spec} k={k}: {len(cos & rawk)} shared ids"


RUNS = [(d, impl, Q, hyb) for d in ("s64", "s768") for impl in IMPLS for Q in (1, 17, 64, 65, 300) for hyb in (0, 1)]


@pytest.mark.parametrize("corpus,impl,Q,hybrid", RUNS, ids=[f"{d}-{i}-Q{q}-{'hyb' if h else 'dense'}"
                                                           for d, i, q, h in RUNS])
def test_cosine_search_exact(corpus, impl, Q, hybrid):
    c = _corpus(corpus)
    Fs = c["Fs"] if hybrid else 0
    r = _retriever(c, n_sparse=Fs)
    specs = _qspecs(Q, c["dim"], salt=Q + hybrid)
    q = torch.from_numpy(_query_rows(specs, c["dim"])).to(DEV)
    kw = {"sparse": _sparse_tensor(c, Q)} if hybrid else {}
    for k in (1, 100, 128):
        s, i = r.search(q, top_k=k, impl=impl, **kw)
        ws, wi = _expected(c, specs, k, c["Fd"], range(Fs), c["Fd"] + Fs, c["base"])
        _assert_exact(s, i, ws, wi, f"{corpus} {impl} Q={Q} hybrid={hybrid} k={k}")


# ---------------------------------------------------------------------------------------------- 3. entry points
def test_search_host_cosine():
    c = _corpus("s768")
    r = _retriever(c, n_sparse=c["Fs"])
    for Q, impl in ((17, "tcgen05"), (129, "auto")):
        specs = _qspecs(Q, c["dim"], salt=5)
        qh = r.corpus.prepare_queries(torch.from_numpy(_query_rows(specs, c["dim"]))).cpu().pin_memory()
        sp = _sparse_tensor(c, Q)[:, :, :c["N"]].cpu().contiguous()
        for k in (2, 128):
            s, i = r.search_host(qh, None, sp, top_k=k, impl=impl)
            ws, wi = _expected(c, specs, k, c["Fd"], range(c["Fs"]), c["Fd"] + c["Fs"], c["base"])
            _assert_exact(s, i, ws, wi, f"search_host Q={Q} k={k}")


def test_graphed_search_fp32_host_queries():
    """Host fp32 queries whose rounding to bf16 BEFORE the normalisation changes the unit row: the graph must round once,
    after it, as the eager search does."""
    GraphedSearch, _, _, _ = _mods()
    c = _corpus("s768")
    r = _retriever(c, n_sparse=c["Fs"])
    Q, k = 64, 100
    g = GraphedSearch(r, Q, sparse="dense", top_k=k)
    for salt in (0, 9):
        specs = _qspecs(Q, c["dim"], salt)
        q = torch.from_numpy(_query_rows(specs, c["dim"]))
        s, i = g(q, None, _sparse_tensor(c, Q))
        ws, wi = _expected(c, specs, k, c["Fd"], range(c["Fs"]), c["Fd"] + c["Fs"], c["base"])
        _assert_exact(s, i, ws, wi, f"GraphedSearch exact salt={salt}")
    # continuous fp32 queries: bf16(q) normalised differs from q normalised in many elements
    gq = torch.Generator().manual_seed(4)
    q = torch.randn(Q, c["dim"], generator=gq) * 3 + 1
    assert not torch.equal(r.corpus.prepare_queries(q), r.corpus.prepare_queries(q.to(torch.bfloat16)))
    sp = _sparse_tensor(c, Q)
    es, ei = r.search(q.to(DEV), sparse=sp, top_k=k)
    gs, gi = g(q, None, sp)
    assert torch.equal(gs.cpu(), es.cpu()) and torch.equal(gi.cpu(), ei.cpu())


def test_mask_sweep_cosine():
    c = _corpus("s768")
    r = _retriever(c, n_sparse=c["Fs"])
    sets = [[], [0], [2], [0, 1], [1, 3]]
    for Q in (17, 257):
        specs = _qspecs(Q, c["dim"], salt=Q)
        q = torch.from_numpy(_query_rows(specs, c["dim"])).to(DEV)
        for k in (1, 128):
            s, i = r.search_mask_sweep(q, sets, sparse=_sparse_tensor(c, Q), top_k=k)
            for m, masked in enumerate(sets):
                dense = sum(1 for f in range(c["Fd"]) if f not in masked)
                sjs = [j for j in range(c["Fs"]) if c["Fd"] + j not in masked]
                ws, wi = _expected(c, specs, k, dense, sjs, c["Fd"] + c["Fs"], c["base"])
                _assert_exact(s[m], i[m], ws, wi, f"mask sweep {masked} Q={Q} k={k}")


def _zero_init(ws, wi):
    neg = ws < 0
    return ws.masked_fill(neg, 0.0), wi.masked_fill(neg, 0)


def _quirk_specs(c, Q):
    """Queries on the whole row (every doc overlaps), half of them negative: those have ~N/61 positive cosines, fewer
    than k, so the (0.0, row 0) initialisation fills the tail."""
    M = _levels(c["dim"])
    specs = [(M, 0, -1 if i % 2 else 1, float(2.0 ** (i * 9 - 30))) for i in range(Q)]
    for sp in specs:
        pos = int((_cos_int(sp, c["lay"]) > 0).sum())
        assert (pos < 100) == (sp[2] < 0)
    return specs


def test_per_field_topk_and_dense_flat_index_cosine():
    from mfar_b200.data.index import DenseFlatIndex
    c = _corpus("s64")
    r = _retriever(c, n_sparse=c["Fs"])
    specs = _qspecs(30, c["dim"], salt=2) + _quirk_specs(c, 10)
    Q = len(specs)
    q = torch.from_numpy(_query_rows(specs, c["dim"]))
    sp = _sparse_tensor(c, Q)
    for k in (2, 100, 128):
        for zero_init in (False, True):
            s, i = r.per_field_topk(q.to(DEV), sp, top_k=k, zero_init=zero_init)
            ws, wi = _expected(c, specs, k, 1, [], 1, 0)
            if zero_init:
                ws, wi = _zero_init(ws, wi)
            for f in range(c["Fd"]):
                _assert_exact(s[f], i[f], ws, wi, f"per_field_topk field {f} k={k} zero_init={zero_init}")
    src = _doc_rows(c["lay"], c["dim"], 0, c["N"])
    keys = [f"d{n}" for n in range(c["N"])]
    idx = DenseFlatIndex(None, src, keys, {kk: n for n, kk in enumerate(keys)}, device=DEV, normalize=True)
    for k in (100, 128):
        got = idx.retrieve_batch(q.numpy(), k)
        ws, wi = _zero_init(*_expected(c, specs, k, 1, [], 1, 0))
        for qi in range(Q):
            assert [kk for kk, _ in got[qi]] == [keys[j] for j in wi[qi].tolist()], f"retrieve_batch q={qi} k={k}"
            assert [v for _, v in got[qi]] == ws[qi].tolist(), f"retrieve_batch scores q={qi} k={k}"
    cand = [keys[j] for j in (0, 3, 64, 1000, 4096, 2048, 5)]
    sb = idx.score_batch(q.numpy(), cand).cpu()
    want = torch.stack([torch.from_numpy(_cos_int(sp_, c["lay"])[[0, 3, 64, 1000, 4096, 2048, 5]] / 256.0).float()
                        for sp_ in specs])
    assert torch.equal(sb, want)


def test_score_candidates_cosine():
    c = _corpus("s768")
    r = _retriever(c, n_sparse=c["Fs"])
    specs = _qspecs(20, c["dim"], salt=3)
    q = torch.from_numpy(_query_rows(specs, c["dim"])).to(DEV)
    rows = torch.tensor([0, 1, 2, 3, 4, 127, 128, 129, 2000, 4096, -1, 77])
    out = r.score_candidates(q, rows, sparse=_sparse_tensor(c, 20)).cpu()
    rw = rows.clamp(min=0).numpy()
    valid = (rows >= 0).float()
    dense = torch.stack([torch.from_numpy(_cos_int(sp, c["lay"])[rw] / 256.0).float() for sp in specs]) * valid
    assert torch.equal(out[0], dense) and torch.equal(out[1], dense)
    for j in range(c["Fs"]):
        want = (torch.from_numpy(c["u"][j][rw] / 256.0).float() * valid).expand(20, -1)
        assert torch.equal(out[c["Fd"] + j], want)


def test_union_rescore_and_trec_eval_step_cosine():
    """Union of the per-field top-k (dense with the (0.0, row 0) entries, sparse) rescored under every field; the
    closed form ranks the union by (score desc, row asc)."""
    c = _corpus("s768")
    r = _retriever(c, n_sparse=c["Fs"], base=0)
    r.numeric_ids_to_keys = [f"d{n}" for n in range(c["N"])]
    specs = _qspecs(24, c["dim"], salt=6)
    Q, k, F = len(specs), 100, c["Fd"] + c["Fs"]
    q = torch.from_numpy(_query_rows(specs, c["dim"])).to(DEV)
    sp = _sparse_tensor(c, Q)
    vals, rows, usize = r.union_rescore_batch(q, sparse=sp, top_k=k)
    ws, wi = np.empty((Q, k), np.float32), np.empty((Q, k), np.int64)
    for qi, spec in enumerate(specs):
        d_s, d_i = _zero_init(*_expected(c, [spec], k, 1, [], 1, 0))
        union = set(d_i[0].tolist())
        for j in range(c["Fs"]):
            union |= set(X.topk_order(c["u"][j], k).tolist())
        U = np.array(sorted(union))
        assert int(usize[qi]) == len(U)
        T = _key(c, spec, c["Fd"], range(c["Fs"]))[U]
        o = X.topk_order(T, k)
        wi[qi], ws[qi] = U[o], (T[o] / (256.0 * F)).astype(np.float32)
    _assert_exact(vals, rows, torch.from_numpy(ws), torch.from_numpy(wi), "union_rescore_batch")
    buf = io.StringIO()
    r.trec_eval_step([f"q{i}" for i in range(Q)], q, buf, sparse=sp, mode="union_rescore")
    lines = [ln.split("\t") for ln in buf.getvalue().splitlines()]
    assert [ln[2] for ln in lines] == [f"d{j}" for j in wi.reshape(-1).tolist()]
    assert [float(ln[4]) for ln in lines] == ws.reshape(-1).tolist()


@pytest.mark.parametrize("Q", [17, 129])
def test_shards_cosine(Q):
    """Window shards (cut inside the pattern's tie groups) merged by ``merge_keys`` and by the virtual-rank exchange,
    and a one-rank ``ShardedRetriever``: all equal the closed form."""
    from mfar_b200.dist import PeerExchange, ShardedRetriever, merge_keys
    c = _corpus("s768")
    cuts = [0, 1280, 2944, c["N"]]
    specs = _qspecs(Q, c["dim"], salt=8)
    q = torch.from_numpy(_query_rows(specs, c["dim"])).to(DEV)
    R = len(cuts) - 1
    for k in (1, 100, 128):
        ws, wi = _expected(c, specs, k, c["Fd"], [], c["Fd"], c["base"])
        parts = []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            sh = _retriever(c, base=c["base"] + lo, top_k=k, pc=c["pc"].window(lo, hi - lo))
            parts.append(sh.search(q, top_k=k, return_keys=True)[2])
        keys = torch.stack(parts)
        s, i = merge_keys(keys, k)
        _assert_exact(s, i, ws, wi, f"merge_keys Q={Q} k={k}")
        s, i = ShardedRetriever(_retriever(c)).search(q, top_k=k)
        _assert_exact(s, i, ws, wi, f"ShardedRetriever Q={Q} k={k}")
        if Q > 17:
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
            _assert_exact(s_r, i_r, ws, wi, f"PeerExchange rank {rk} Q={Q} k={k}")


# ---------------------------------------------------------------------------------------------- 4. mixture default
def test_mixture_default_is_the_normalised_query():
    """With a query-conditioned mixture, q_emb defaults to the unit query on a cosine corpus (the reference's encoder
    ends in Normalize()): search, the sweep, union_rescore and the graph all equal the explicit call."""
    GraphedSearch, MultiFieldRetriever, PackedCorpus, LinearWeights = _mods()
    g = torch.Generator().manual_seed(9)
    N, dim, Fd, Fs, Q, k = 3072, 128, 3, 1, 32, 50      # N % 64 == 0: eager and graph read the same sparse layout
    fields = [torch.randn(N, dim, generator=g) * (f + 1) for f in range(Fd)]
    pc = PackedCorpus.from_fields(fields, DEV, normalize=True)
    layer = LinearWeights(dim, Fd + Fs, query_cond=True)
    with torch.no_grad():
        layer.weight.copy_(torch.randn(dim, Fd + Fs, generator=g))
    r = MultiFieldRetriever(pc, layer.to(DEV), n_sparse=Fs, top_k=k)
    q = (torch.randn(Q, dim, generator=g) * 40).to(DEV)
    sp = (torch.rand(Q, Fs, N, generator=g) * 2).half().to(DEV)
    qn = torch.nn.functional.normalize(q.float(), dim=1)
    a = r.search(q, sparse=sp)
    b = r.search(q, qn, sparse=sp)
    raw = r.search(q, q.float(), sparse=sp)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert not torch.equal(raw[1], b[1]), "raw and unit q_emb give the same ranking: the check is vacuous"
    a = r.search_mask_sweep(q, [[], [1]], sparse=sp)
    b = r.search_mask_sweep(q, [[], [1]], q_emb=qn, sparse=sp)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    a = r.union_rescore_batch(q, sparse=sp)
    b = r.union_rescore_batch(q, qn, sparse=sp)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    gs = GraphedSearch(r, Q, sparse="dense", top_k=k)
    ref = r.search(q, qn, sparse=sp, top_k=k)
    s, i = gs(q.cpu(), None, sp)
    assert torch.equal(s, ref[0]) and torch.equal(i, ref[1])
    s, i = gs(q, qn, sp)
    assert torch.equal(s, ref[0]) and torch.equal(i, ref[1])


# ---------------------------------------------------------------------------------------------- 5. at scale
# (impl, Q, {k: threshold-seeding prefix levels}); every prefix level adds 4 launches (csrc/capi.cu)
SCALE = [("tcgen05", 40, {1: 1, 100: 2}), ("auto", 300, {100: 2})]


@pytest.mark.parametrize("impl,Q,levels", SCALE, ids=[f"{i}-Q{q}" for i, q, _ in SCALE])
def test_cosine_search_at_scale(impl, Q, levels):
    """4M ragged docs packed in the default chunks from a host fp32 array; magnitudes 2^-36 .. 2^70 across the corpus."""
    c = _corpus("l4m")
    r = _retriever(c)
    specs = _qspecs(Q, c["dim"], salt=Q)
    q = torch.from_numpy(_query_rows(specs, c["dim"])).to(DEV)
    for k, lv in levels.items():
        s, i = r.search(q, top_k=k, impl=impl)
        assert r.last_launches == 2 + 4 * lv, f"k={k}: {r.last_launches} launches, want {lv} prefix levels"
        ws, wi = _expected(c, specs, k, 1, [], 1, c["base"])
        _assert_exact(s, i, ws, wi, f"l4m {impl} Q={Q} k={k}")


def test_zz_release_hbm():
    _free()
