"""NaN and +-inf scores on every scoring path against a closed-form answer, compared with ``torch.equal``.

The inputs are tests/exact_nonfinite.py: exact_topk's integer patterns plus NaN and +inf planted on reserved
coordinates, so a query's coefficients (+1, -1, 0) make the same docs score +inf, -inf or NaN; sparse rows add +-inf
and NaN of both signs per query.  The rule every ranked path follows (csrc/common.cuh, ``mfar_oracle.rank_rows``):
NaN (any sign or payload) > +inf > finite scores descending > -inf, the lower doc id first inside a class; a NaN doc
reports a NaN score, infinite docs report +-inf with their ids, and since k <= N no slot is ever (-inf, -1).  A
query's answer does not depend on the other queries of its batch (asserted directly in test_batch_invariance).
"""
import gc

import numpy as np
import pytest
import torch

import exact_nonfinite as NF
import exact_topk as X
import mfar_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda"
IMPLS = ("simt", "tcgen05", "tcgen05_qs", "auto")
KS = (1, 100, 128)
TOP = 2 ** 32

# name: (N, dim, dense fields, sparse fields, doc_id_base, planted, almost-all plant)
CORPORA = {
    "s4097": (4097, 768, 2, 2, TOP - 4097, True, False),
    "s4097_almost": (4097, 768, 1, 0, TOP - 4097, True, True),
    "c4097": (4097, 768, 2, 2, TOP - 4097, False, False),     # clean dense rows: non-finite scores from sparse rows only
    "m330k": (330_001, 768, 2, 2, TOP - 330_001, True, False),
    "l4m": (4_000_001, 64, 1, 0, TOP - 4_000_001, True, False),
}
_cache = {}


def _free():
    _cache.clear()
    _ranked.clear()
    gc.collect()
    torch.cuda.empty_cache()


def _corpus(name):
    if name in _cache:
        return _cache[name]
    if name in ("m330k", "l4m"):                         # one large corpus at a time
        for other in ("m330k", "l4m"):
            _cache.pop(other, None)
        _ranked.clear()
        gc.collect()
        torch.cuda.empty_cache()
    from mfar_b200.modeling.retrieval import PackedCorpus
    N, dim, Fd, Fs, base, planted, almost = CORPORA[name]
    pc = PackedCorpus(N, Fd, dim, DEV)
    docs = X.doc_matrix(N, dim)
    cols = NF.plant_columns(N, dim, almost) if planted else {}
    for lo in range(0, N, 1 << 18):
        hi = min(N, lo + (1 << 18))
        rows = torch.from_numpy(docs[lo:hi]).to(DEV).to(torch.bfloat16)
        bits = rows.view(torch.int16)
        for p, v in cols.items():
            sel = torch.from_numpy(v[lo:hi]).to(DEV)
            bits[:, p] = torch.where(sel != 0, sel, bits[:, p])
        for f in range(Fd):
            pc.load_rows(f, lo, rows)
    n = np.arange(N, dtype=np.int64)
    u = np.stack([(n // 7) % 11 * 64, np.where(n % 1009 == 5, 2048, (n * 13) % 17)])[:Fs].astype(np.float64)
    c = dict(pc=pc, N=N, dim=dim, Fd=Fd, Fs=Fs, base=base, planted=planted, almost=almost, u=u, dense={})
    _cache[name] = c
    return c


def _coefs(c, i, salt):
    if not c["planted"]:
        return ()
    if c["almost"]:
        cf = [cb + (a,) for cb in NF.COEFS for a in (1, -1, 0)]
        return cf[(i * 5 + salt) % len(cf)]
    return NF.COEFS[(i * 5 + salt) % len(NF.COEFS)]


def _spec(c, Q, salt):
    """Per query: (pattern combo, plant coefficients)."""
    return [(X.COMBOS[(i * 7 + salt) % len(X.COMBOS)], _coefs(c, i, salt)) for i in range(Q)]


def _queries(c, spec):
    return torch.from_numpy(np.stack([NF.query_vector(cb, cf, c["dim"]) for cb, cf in spec])).to(DEV)


def _dense(c, cb, cf):
    """float64 [N] dot product of a query with every doc (cached)."""
    key = (cb, cf)
    if key not in c["dense"]:
        if c["planted"]:
            c["dense"][key] = NF.dense_values(cb, cf, c["N"], c["almost"])
        else:
            c["dense"][key] = X.dense_scores(*cb, c["N"]).astype(np.float64)
    return c["dense"][key]


_ranked = {}                                           # id(float64 row) -> (row, top-128 order, fp32 row)


def _want(scores64, k, base, memo=False):
    """Expected (scores fp32 [Q,k], ids int64 [Q,k]) from float64 exact scores [Q rows of N]: the top 128 of every
    distinct row object is ranked once (the order is total, so the top k is its prefix); ``memo``: the rows are the
    cached ones of ``_dense`` and their rankings are kept across calls."""
    Q = len(scores64)
    ws = np.empty((Q, k), dtype=np.float32)
    wi = np.empty((Q, k), dtype=np.int64)
    ranked = _ranked if memo else {}
    for q, s in enumerate(scores64):
        hit = ranked.get(id(s))
        if hit is None or hit[0] is not s:
            s32 = s.astype(np.float32)
            hit = ranked[id(s)] = (s, O.rank_rows(s32, 128), s32)
        _, o, s32 = hit
        ws[q], wi[q] = s32[o[:k]], o[:k] + base
    return torch.from_numpy(ws), torch.from_numpy(wi)


def _same(a, b):
    """Exact equality with NaN == NaN (any payload)."""
    a, b = a.cpu(), b.cpu()
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a[~na], b[~nb])


def _assert_exact(s, i, want_s, want_i, what):
    s, i = s.cpu(), i.cpu()
    assert not bool((i < 0).any()), f"{what}: an empty (-inf, -1) slot with k <= N"
    if torch.equal(i, want_i) and _same(s, want_s):
        return
    bad = [q for q in range(want_i.shape[0]) if not (torch.equal(i[q], want_i[q]) and _same(s[q], want_s[q]))]
    q = bad[0]
    if torch.equal(i[q], want_i[q]):
        j = int(((torch.isnan(s[q]) != torch.isnan(want_s[q])) | ((s[q] != want_s[q]) & ~torch.isnan(want_s[q])))
                .nonzero()[0])
    else:
        j = int((i[q] != want_i[q]).nonzero()[0])
    raise AssertionError(f"{what}: {len(bad)} of {want_i.shape[0]} queries wrong, first q={q} rank {j}: "
                         f"got ({s[q, j].item()}, {i[q, j].item()}), want ({want_s[q, j].item()}, {want_i[q, j].item()})")


def _retriever(c, n_sparse=0, base=None, top_k=100):
    from mfar_b200.modeling.retrieval import MultiFieldRetriever
    from mfar_b200.modeling.weighting import LinearWeights
    F = c["Fd"] + n_sparse
    layer = LinearWeights(F, 1).to(DEV)                 # equal static logits: weights exactly 1/F
    r = MultiFieldRetriever(c["pc"], layer, n_sparse=n_sparse, top_k=top_k,
                            doc_id_base=c["base"] if base is None else base)
    w = layer.field_weights(None, r.mask, batch=1)
    assert torch.equal(w, torch.full((1, F), 1.0 / F, device=DEV)), "mixture weights are not exactly 1/F"
    return r


def _launches(levels, extra=0):
    return 2 + 4 * levels + extra


def _dense_only(c, spec):
    """Dense-only mixture (Fd identical fields at weight 1/Fd): the dot product itself."""
    return [_dense(c, cb, cf) for cb, cf in spec]


# ---------------------------------------------------------------------------------------------- dense search
QS = (1, 7, 8, 9, 64, 129, 512)
SMALL_RUNS = [(c, impl, Q) for c in ("s4097", "s4097_almost") for impl in IMPLS for Q in QS]


@pytest.mark.parametrize("corpus,impl,Q", SMALL_RUNS, ids=[f"{c}-{i}-Q{q}" for c, i, q in SMALL_RUNS])
def test_search_dense_nonfinite(corpus, impl, Q):
    """NaN docs (both signs), +-inf and 0 * inf = NaN docs, +inf + -inf = NaN where plants overlap; with the almost-all
    plant at coefficient -1 fewer than k docs score above -inf and the rest of the list is real -inf docs."""
    c = _corpus(corpus)
    r = _retriever(c)
    spec = _spec(c, Q, salt=Q)
    q = _queries(c, spec)
    want64 = _dense_only(c, spec)
    for k in KS:
        s, i = r.search(q, top_k=k, impl=impl)
        assert r.last_launches == _launches(0)
        ws, wi = _want(want64, k, c["base"], memo=True)
        _assert_exact(s, i, ws, wi, f"{corpus} {impl} Q={Q} k={k}")


# (impl, Q, {k: expected prefix levels}) as in test_gpu_topk_exact.py; the ``many`` plant puts >= 128 +inf / -inf /
# NaN docs (by the query's coefficient) inside the one-tile-per-CTA prefix of the seeded runs
MID_RUNS = [("simt", 1, {1: 0, 100: 0, 128: 0}), ("tcgen05", 1, {1: 0, 128: 0}), ("tcgen05_qs", 1, {100: 0}),
            ("auto", 9, {100: 0}), ("tcgen05", 32, {1: 1, 100: 1}), ("tcgen05", 129, {1: 1, 100: 2}),
            ("tcgen05_qs", 33, {100: 1}), ("tcgen05_qs", 257, {2: 1, 100: 2}), ("auto", 64, {100: 1}),
            ("auto", 512, {2: 1, 100: 2, 127: 2})]
LARGE_RUNS = [("simt", 1, {100: 0}), ("tcgen05", 1, {1: 0, 128: 0}), ("tcgen05_qs", 7, {100: 0}),
              ("tcgen05", 64, {2: 1, 128: 2}), ("tcgen05_qs", 64, {1: 1, 100: 2}), ("auto", 129, {100: 2}),
              ("tcgen05", 512, {1: 2, 100: 2})]
BIG = [("m330k",) + r for r in MID_RUNS] + [("l4m",) + r for r in LARGE_RUNS]


@pytest.mark.parametrize("corpus,impl,Q,levels", BIG, ids=[f"{c}-{i}-Q{q}" for c, i, q, _ in BIG])
def test_search_at_scale_nonfinite(corpus, impl, Q, levels):
    c = _corpus(corpus)
    r = _retriever(c)
    spec = _spec(c, Q, salt=3 * Q + 1)
    q = _queries(c, spec)
    want64 = _dense_only(c, spec)
    for k, lv in levels.items():
        s, i = r.search(q, top_k=k, impl=impl)
        assert r.last_launches == _launches(lv), f"k={k}: {r.last_launches} launches, want {lv} prefix levels"
        ws, wi = _want(want64, k, c["base"], memo=True)
        _assert_exact(s, i, ws, wi, f"{corpus} {impl} Q={Q} k={k}")


# ---------------------------------------------------------------------------------------------- sparse rows
SPARSE_MODES = ("fin", "mix", "allnan", "ninf")


def _sparse_values(c, mode):
    """float64 [Fs, N] sparse scores of one query: exact_topk-style integers plus the mode's non-finite plants.
    ``mix``: +inf, -inf, +NaN in field 0, -NaN and +inf in field 1 - the +inf at doc 3, a ``many`` doc, so a query
    with coefficient -1 there scores -inf + inf = NaN; ``allnan``: every doc NaN; ``ninf``: -inf at every doc but ~40."""
    N = c["N"]
    n = np.arange(N)
    u = c["u"].copy()
    if mode == "mix":
        u[0, n % 211 == 17] = np.inf
        u[0, n % 211 == 50] = -np.inf
        u[0, n % 211 == 90] = np.nan
        u[1, n % 307 == 11] = NF.NEG_NAN_F32
        u[1, 3] = np.inf
    elif mode == "allnan":
        u[:] = np.nan
    elif mode == "ninf":
        u[0, n % max(2, N // 40) != 1] = -np.inf
    return u


def _hybrid_spec(c, Q, salt, modes=SPARSE_MODES):
    spec = _spec(c, Q, salt)
    out = []
    for i, (cb, cf) in enumerate(spec):
        mode = modes[(i * 3 + salt) % len(modes)]
        if mode == "ninf" and c["planted"]:
            cf = (-1, -1)                              # few and many at -inf too: fewer than k docs above -inf
        if mode == "mix" and c["planted"] and i % 2 == 0:
            cf = (cf[0], -1)                           # dense -inf + sparse +inf at doc 3
        out.append((cb, cf, mode))
    return out


def _hybrid_want(c, hspec, F):
    out = []
    for cb, cf, mode in hspec:
        sp = _sparse_values(c, mode).astype(np.float32).astype(np.float64)   # what f16 / f32 rows hold (all exact)
        with np.errstate(invalid="ignore"):
            out.append((c["Fd"] * _dense(c, cb, cf) + sp.sum(axis=0)) / F)
    return out


def _to_f16(x):
    """float32 -> float16 keeping the sign bit of NaNs (numpy's cast drops it)."""
    h = x.astype(np.float16)
    h.view(np.uint16)[np.isnan(x) & np.signbit(x)] |= np.uint16(0x8000)
    return h


def _sparse_np(c, hspec, f32):
    rows = np.stack([_sparse_values(c, m) for _, _, m in hspec]).astype(np.float32)
    return rows if f32 else _to_f16(rows)


def _sparse_tensor(c, hspec, dtype, ld=None):
    N = c["N"]
    ld = ld or (N + 63) // 64 * 64
    rows = _sparse_np(c, hspec, dtype == torch.float32)
    sp = torch.zeros((len(hspec), c["Fs"], ld), dtype=dtype, device=DEV)
    ity = torch.int32 if dtype == torch.float32 else torch.int16
    sp.view(ity)[:, :, :N] = torch.from_numpy(rows).to(DEV).view(ity)      # copied as integers: bit exact
    return sp


def _coo(c, hspec):
    rows = torch.from_numpy(_sparse_np(c, hspec, False)).to(DEV)         # [Q, Fs, N] f16
    keys, vals, off = [], [], [0]
    for j in range(c["Fs"]):
        nz = (rows[:, j] != 0) | torch.isnan(rows[:, j])
        qq, dd = nz.nonzero(as_tuple=True)
        keys.append(torch.stack([qq.int(), dd.int()], dim=1))
        vals.append(rows.view(torch.int16)[qq, j, dd].view(torch.float16))      # gathered as integers: bit exact
        off.append(off[-1] + int(qq.numel()))
    return torch.cat(keys).contiguous(), torch.cat(vals).contiguous(), off


SPARSE_RUNS = [(c, i, q, lay) for c, i, q in
               [("s4097", "tcgen05", Q) for Q in (1, 9, 64)] + [("s4097", "auto", Q) for Q in (65, 512)] +
               [("s4097", "simt", 33), ("s4097", "tcgen05_qs", 8), ("m330k", "tcgen05", 64), ("m330k", "auto", 512)]
               for lay in ("f16_aligned", "f16_unaligned", "f32", "coo")
               if not (lay == "coo" and c == "m330k")]


@pytest.mark.parametrize("corpus,impl,Q,layout", SPARSE_RUNS, ids=[f"{c}-{i}-Q{q}-{l}" for c, i, q, l in SPARSE_RUNS])
def test_search_sparse_layouts_nonfinite(corpus, impl, Q, layout):
    """Planted dense rows plus sparse rows with +-inf, NaN of both signs, an all-NaN row and an almost-all -inf row, in
    every sparse layout: fused f16 rows, an unaligned pitch (pre-mix kernel), f32 rows and COO pairs."""
    c = _corpus(corpus)
    base = 0 if layout == "coo" else c["base"]
    r = _retriever(c, n_sparse=c["Fs"], base=base)
    hspec = _hybrid_spec(c, Q, salt=Q)
    q = _queries(c, [(cb, cf) for cb, cf, _ in hspec])
    F = c["Fd"] + c["Fs"]
    want64 = _hybrid_want(c, hspec, F)
    if layout == "coo":
        kw = dict(sparse_coo=_coo(c, hspec))
    else:
        dtype = torch.float32 if layout == "f32" else torch.float16
        kw = dict(sparse=_sparse_tensor(c, hspec, dtype, c["N"] + 3 if layout == "f16_unaligned" else None))
        # negative NaNs are planted, and the device rows hold exactly the host bits (checked as integers: the sign of
        # a NaN does not survive torch's f16 -> fp32 conversions on the device, e.g. inside torch.signbit)
        host = _sparse_np(c, hspec, dtype == torch.float32)
        assert bool((np.isnan(host) & np.signbit(host)).any()) == any(m == "mix" for *_, m in hspec)
        ity = torch.int32 if dtype == torch.float32 else torch.int16
        assert torch.equal(kw["sparse"].view(ity)[:, :, :c["N"]].cpu(), torch.from_numpy(host).view(ity))
    for k in KS:
        s, i = r.search(q, top_k=k, impl=impl, **kw)
        ws, wi = _want(want64, k, base)
        _assert_exact(s, i, ws, wi, f"{corpus} {layout} {impl} Q={Q} k={k}")


# ---------------------------------------------------------------------------------------------- batch invariance
def _run(r, c, hspec, k, impl, sparse):
    q = _queries(c, [(cb, cf) for cb, cf, _ in hspec])
    kw = dict(sparse=_sparse_tensor(c, hspec, torch.float16)) if sparse else {}
    return r.search(q, top_k=k, impl=impl, **kw)


INV_RUNS = [(c, impl) for c in ("c4097", "s4097", "m330k") for impl in IMPLS]


@pytest.mark.parametrize("corpus,impl", INV_RUNS, ids=[f"{c}-{i}" for c, i in INV_RUNS])
def test_batch_invariance(corpus, impl):
    """Every target query's row equals the same query run alone, inside a batch of mates whose scores are all finite
    (clean dense rows, finite sparse rows) and inside a batch of mates whose scores are all NaN; on planted rows the
    mates take every coefficient, and the targets sit in different groups of 8 and query tiles."""
    c = _corpus(corpus)
    sparse = True
    r = _retriever(c, n_sparse=c["Fs"])
    targets = _hybrid_spec(c, 6, salt=1, modes=("mix", "ninf"))
    mates_fin = [(cb, cf, "fin") for cb, cf, _ in _hybrid_spec(c, 80, salt=4, modes=("fin",))]
    mates_nan = [(cb, cf, "allnan") for cb, cf, _ in _hybrid_spec(c, 80, salt=7, modes=("allnan",))]
    F = c["Fd"] + c["Fs"]
    for k in (1, 100):
        alone = [_run(r, c, [t], k, impl, sparse) for t in targets]
        want = _want(_hybrid_want(c, targets, F), k, c["base"])
        for t in range(len(targets)):
            _assert_exact(alone[t][0], alone[t][1], want[0][t:t + 1], want[1][t:t + 1], f"{corpus} {impl} alone t={t}")
        for name, mates in (("finite mates", mates_fin), ("NaN mates", mates_nan)):
            for Q, where in ((9, (0, 4, 8, 1, 5, 7)), (70, (3, 33, 66, 10, 40, 69))):
                batch = list(mates[:Q])
                for t, w in enumerate(where):
                    batch[w] = targets[t]
                s, i = _run(r, c, batch, k, impl, sparse)
                for t, w in enumerate(where):
                    assert torch.equal(i[w].cpu(), alone[t][1][0].cpu()) and _same(s[w], alone[t][0][0]), \
                        f"{corpus} {impl} k={k} {name} Q={Q}: target {t} at row {w} differs from the same query alone"


# ---------------------------------------------------------------------------------------------- sparse-only rows
def _row_values(combo, i, N, f32):
    """Per-query sparse-only row: pattern integers plus non-finite plants; query 2 of a batch is all NaN, query 3
    -inf at every doc but ~40."""
    name, sign = combo
    if not f32 and name in ("n", "perm", "div37"):
        name = "mod127"                                 # values above 2048 are not exact in f16
    v = X.dense_scores(name, sign, N).astype(np.float32)
    n = np.arange(N)
    if i % 4 == 2:
        v[:] = np.nan
        v[n % 2 == 1] = NF.NEG_NAN_F32
    elif i % 4 == 3:
        v[n % max(2, N // 40) != 1] = -np.inf
    else:
        v[n % 97 == 3 + i % 5] = np.inf
        v[n % 89 == 7] = -np.inf
        v[n % 131 == 11] = np.nan
        v[n % 173 == 19] = NF.NEG_NAN_F32
    return v


@pytest.mark.parametrize("N", [4097, 330_001])
@pytest.mark.parametrize("dtype", ["f16", "f32"])
@pytest.mark.parametrize("Q", [1, 4, 17, 64])
def test_sparse_only_rows_nonfinite(N, dtype, Q):
    """The streaming row top-k of a sparse-only scorer, with its threshold seed (N >= 4096): an all-NaN row returns the
    first k ids, an almost-all -inf row fills its tail with the lowest -inf ids."""
    from mfar_b200.modeling.retrieval import MultiFieldRetriever
    from mfar_b200.modeling.weighting import LinearWeights
    base = TOP - N
    r = MultiFieldRetriever(None, LinearWeights(1, 1).to(DEV), n_sparse=1, top_k=100, n_docs=N, device=DEV,
                            doc_id_base=base)
    f32 = dtype == "f32"
    rows = np.stack([_row_values(X.COMBOS[(i * 7 + Q) % len(X.COMBOS)], i, N, f32) for i in range(Q)])
    rows_t = rows if f32 else _to_f16(rows)
    assert bool((np.isnan(rows_t) & np.signbit(rows_t)).any()), "negative NaNs are planted in every row"
    sp = torch.from_numpy(rows_t).to(DEV).unsqueeze(1).contiguous()
    for k in KS:
        s, i = r.search(None, sparse=sp, top_k=k, batch=Q)
        assert r.last_launches == 4
        ws, wi = _want(list(rows_t.astype(np.float64)), k, base)
        _assert_exact(s, i, ws, wi, f"rows N={N} {dtype} Q={Q} k={k}")
        if Q > 2:
            assert torch.equal(i[2].cpu(), torch.arange(k) + base)


# ---------------------------------------------------------------------------------------------- other entry points
@pytest.mark.parametrize("corpus", ["s4097", "m330k"])
def test_per_field_topk_nonfinite(corpus):
    """Each field ranked alone (weight 1).  With the (0.0, row 0) initialisation negative entries, -inf included, become
    (0.0, row 0); NaN entries outrank the initial zeros under torch.topk's order and stay."""
    c = _corpus(corpus)
    r = _retriever(c, n_sparse=c["Fs"])
    Q = 40
    hspec = _hybrid_spec(c, Q, salt=13)
    q = _queries(c, [(cb, cf) for cb, cf, _ in hspec])
    sp = _sparse_tensor(c, hspec, torch.float16)
    dense64 = [_dense(c, cb, cf) for cb, cf, _ in hspec]
    sparse64 = [_sparse_values(c, m).astype(np.float16).astype(np.float64) for *_, m in hspec]
    for k in (2, 100, 128):
        for zero_init in (False, True):
            s, i = r.per_field_topk(q, sp, top_k=k, zero_init=zero_init)
            ws, wi = _want(dense64, k, 0)
            if zero_init:
                neg = ws < 0
                ws, wi = ws.masked_fill(neg, 0.0), wi.masked_fill(neg, 0)
            for f in range(c["Fd"]):
                _assert_exact(s[f], i[f], ws, wi, f"per_field_topk field {f} k={k} zero_init={zero_init}")
            for j in range(c["Fs"]):
                ws_j, wi_j = _want([x[j] for x in sparse64], k, 0)
                _assert_exact(s[c["Fd"] + j], i[c["Fd"] + j], ws_j, wi_j, f"per_field_topk sparse {j} k={k}")


def test_score_candidates_nonfinite():
    """Per-field scores of chosen rows: every value in its IEEE class (NaN, +-inf), finite ones exact."""
    c = _corpus("s4097")
    r = _retriever(c, n_sparse=c["Fs"])
    Q = 27
    hspec = _hybrid_spec(c, Q, salt=2)
    q = _queries(c, [(cb, cf) for cb, cf, _ in hspec])
    sp = _sparse_tensor(c, hspec, torch.float32)
    S = NF.plant_sets(c["N"])
    rows = np.unique(np.r_[np.nonzero(S["nan"] | S["few"])[0], np.nonzero(S["many"])[0][:40], 3, 17, 50, 90, 11,
                          np.arange(0, c["N"], 97)])
    out = r.score_candidates(q, torch.from_numpy(rows).to(DEV), sp).cpu()
    for f in range(c["Fd"]):
        want = torch.from_numpy(np.stack([_dense(c, cb, cf)[rows] for cb, cf, _ in hspec]).astype(np.float32))
        assert _same(out[f], want), f"dense field {f}"
        assert bool(torch.isnan(want).any() and torch.isinf(want).any())
    for j in range(c["Fs"]):
        want = torch.from_numpy(np.stack([_sparse_values(c, m)[j][rows] for *_, m in hspec]).astype(np.float32))
        assert _same(out[c["Fd"] + j], want), f"sparse field {j}"


def test_union_rescore_nonfinite():
    """Per-field top-k (with the (0.0, row 0) initialisation) -> union -> rescore -> mixture -> top-k, the union
    ranked under the rule."""
    c = _corpus("s4097")
    r = _retriever(c, n_sparse=c["Fs"])
    Q, k = 24, 100
    hspec = _hybrid_spec(c, Q, salt=5)
    q = _queries(c, [(cb, cf) for cb, cf, _ in hspec])
    sp = _sparse_tensor(c, hspec, torch.float16)
    vals, rows, usize = r.union_rescore_batch(q, None, sp, top_k=k)
    F = c["Fd"] + c["Fs"]
    mix64 = _hybrid_want(c, hspec, F)
    for qi, (cb, cf, mode) in enumerate(hspec):
        lists = []
        d = _dense(c, cb, cf).astype(np.float32)
        for f in range(c["Fd"]):
            o = O.rank_rows(d, k)
            o = np.where(d[o] < 0, 0, o)                # (0.0, row 0) initialisation
            lists.append(o)
        spv = _sparse_values(c, mode).astype(np.float16).astype(np.float32)
        for j in range(c["Fs"]):
            lists.append(O.rank_rows(spv[j], k))
        union = np.unique(np.concatenate(lists))
        assert int(usize[qi]) == union.size, f"q={qi}: union of {int(usize[qi])} rows, want {union.size}"
        m = mix64[qi][union].astype(np.float32)
        o = O.rank_rows(m, k)
        want_i = torch.from_numpy(union[o].astype(np.int64))
        want_s = torch.from_numpy(m[o])
        _assert_exact(vals[qi:qi + 1], rows[qi:qi + 1], want_s[None], want_i[None], f"union_rescore q={qi} {mode}")


# ---------------------------------------------------------------------------------------------- merge and exchange
def _merge_lists(L, Q, k_in, seed):
    from mfar_b200.dist import encode_keys
    g = np.random.default_rng(seed)
    scores = g.integers(-20, 20, (L, Q, k_in)).astype(np.float32)
    u = g.random((L, Q, k_in))
    nans = np.array([np.nan, -np.nan, NF.NEG_NAN_F32, np.array([0x7F800001], np.uint32).view(np.float32)[0]],
                    dtype=np.float32)
    scores[u < 0.15] = nans[g.integers(0, 4, int((u < 0.15).sum()))]
    scores[(u >= 0.15) & (u < 0.3)] = np.inf
    scores[(u >= 0.3) & (u < 0.45)] = -np.inf
    ids = g.permutation(L * Q * k_in).reshape(L, Q, k_in).astype(np.int64) * 3 + 7
    return scores, ids, encode_keys(scores, ids)


def _merge_want(scores, ids, k):
    L, Q, k_in = scores.shape
    s = scores.transpose(1, 0, 2).reshape(Q, -1)
    i = ids.transpose(1, 0, 2).reshape(Q, -1)
    ws = np.empty((Q, k), dtype=np.float32)
    wi = np.empty((Q, k), dtype=np.int64)
    for q in range(Q):                                   # rank by (class, score, id asc): sort on ids first
        perm = np.argsort(i[q], kind="stable")
        o = perm[O.rank_rows(s[q][perm], k)]
        ws[q], wi[q] = s[q][o], i[q][o]
    return torch.from_numpy(ws), torch.from_numpy(wi)


@pytest.mark.parametrize("L,Q,k_in", [(12, 5, 128), (320, 3, 128), (3, 4, 100)])
def test_merge_keys_nonfinite(L, Q, k_in):
    """``mfar_topk_merge`` over keys from ``encode_keys`` holding NaN of both signs and payloads and +-inf: NaN keys form
    one class above +inf, ranked by id."""
    from mfar_b200.dist import merge_keys
    scores, ids, keys = _merge_lists(L, Q, k_in, seed=L + Q)
    dev = torch.from_numpy(keys.view(np.int64)).to(DEV)
    for k in (1, 100, 128):
        s, i = merge_keys(dev, k)
        ws, wi = _merge_want(scores, ids, k)
        _assert_exact(s, i, ws, wi, f"merge_keys L={L} Q={Q} k={k}")


def test_exchange_nonfinite():
    """The peer exchange + merge with virtual ranks on one device, over the same kind of keys."""
    from mfar_b200.dist import PeerExchange
    R, Q, k_in = 3, 9, 128
    scores, ids, keys = _merge_lists(R, Q, k_in, seed=5)
    dev = torch.from_numpy(keys.view(np.int64)).to(DEV)
    n = PeerExchange.buffer_bytes(R, 256, 128)
    bufs = [torch.zeros(n, dtype=torch.uint8, device=DEV) for _ in range(R)]
    ex = [PeerExchange(256, 128, peer_buffers=bufs, rank=rk, world=R) for rk in range(R)]
    streams = [torch.cuda.Stream() for _ in range(R)]
    for k in (1, 128):
        torch.cuda.synchronize()
        outs = []
        for rk in range(R):
            with torch.cuda.stream(streams[rk]):
                outs.append(ex[rk].merge(dev[rk].contiguous(), k))
        torch.cuda.synchronize()
        ws, wi = _merge_want(scores, ids, k)
        for rk, (s_r, i_r) in enumerate(outs):
            _assert_exact(s_r, i_r, ws, wi, f"PeerExchange rank {rk} k={k}")


# ---------------------------------------------------------------------------------------------- dense overflow
def test_dense_overflow():
    """Finite bf16 inputs whose product overflows fp32: doc coordinate 2^100 times query coefficient +-2^100 on a
    reserved coordinate.  Every implementation gives the IEEE result (+-inf; 0 for a zero coefficient), and a query's
    answer does not depend on its batch."""
    from mfar_b200.modeling.retrieval import PackedCorpus, MultiFieldRetriever
    from mfar_b200.modeling.weighting import LinearWeights
    N, dim = 4097, 768
    big = NF.reserved(dim)["big"]
    docs = torch.from_numpy(X.doc_matrix(N, dim)).to(torch.float32)
    n = np.arange(N)
    S_big = (n % 61 == 5) | (n < 3)
    docs[torch.from_numpy(S_big), big] = 2.0 ** 100
    pc = PackedCorpus(N, 1, dim, DEV)
    pc.load_rows(0, 0, docs.to(DEV).to(torch.bfloat16))
    r = MultiFieldRetriever(pc, LinearWeights(1, 1).to(DEV), top_k=100, doc_id_base=0)
    Q = 24
    combos = [X.COMBOS[(i * 7) % len(X.COMBOS)] for i in range(Q)]
    cbig = [(1, -1, 0)[i % 3] for i in range(Q)]
    qv = np.stack([X.query_vector(*cb, dim) for cb in combos])
    qv[:, big] = np.array(cbig, dtype=np.float32) * np.float32(2.0 ** 100)
    q = torch.from_numpy(qv).to(DEV)
    want64 = []
    for cb, cc in zip(combos, cbig):
        v = X.dense_scores(*cb, N).astype(np.float64)
        v[S_big] = v[S_big] + (cc * np.inf if cc else 0.0)
        want64.append(v)
    for impl in IMPLS:
        for k in KS:
            s, i = r.search(q, top_k=k, impl=impl)
            ws, wi = _want(want64, k, 0)
            _assert_exact(s, i, ws, wi, f"overflow {impl} k={k}")
            s1, i1 = r.search(q[1:2], top_k=k, impl=impl)
            assert torch.equal(i1.cpu(), i[1:2].cpu()) and _same(s1, s[1:2]), f"overflow {impl} k={k}: batch-dependent"


def test_zz_release_hbm():
    _free()
