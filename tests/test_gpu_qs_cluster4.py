"""Large-batch kernel in 4-CTA clusters: the two CTA pairs of a worker column share every doc tile by TMA multicast.

The kernel is launched with a preferred cluster of 4 where the query tiles come in fours and a stage splits into two
K halves; each case here checks the ranked top-k against the fp32 checker (tests/checker.py) and that 4-CTA clusters
actually ran (mfar_profile_cluster4_ctas) - or, for a dim whose stage has an odd chunk count, that none did.
"""
import gc

import pytest
import torch

import mfar_oracle as O
from checker import Fp32Checker, assert_topk_parity_at_scale
from parity import assert_topk_parity

pytestmark = pytest.mark.gpu

DEV = "cuda"
K = 100


def _cluster4_ctas():
    from mfar_b200 import _native as nv
    n = nv.lib().mfar_profile_cluster4_ctas()
    assert n >= 0
    return n


def _retriever(n, F, d, Q, seed):
    from mfar_b200 import synth as S
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    pc = PackedCorpus(n, F, d, DEV)
    S.fill_packed_corpus(pc, seed=seed)
    q = S.make_queries(Q, d, S.corpus_mean(d, seed, DEV), seed + 1, DEV)
    layer = LinearWeights(d, F, query_cond=True)
    with torch.no_grad():
        layer.weight.copy_(S.make_mixture(d, F, seed + 2))
    r = MultiFieldRetriever(pc, layer.to(DEV), top_k=K)
    w = O.mixture_weights(q.float().cpu(), layer.weight.detach().cpu(), True).to(DEV)
    return r, pc, q, w


# (n_docs, dense fields, dim, Q, seed, 4-CTA clusters expected).  37 workers at Q > 384: threshold seeding starts at
# 592 tiles (75.8k docs) and takes its second level above ~168k docs; every n_docs leaves a ragged last tile.
CASES = {
    "q512_unseeded": (50_001, 3, 768, 512, 41, True),
    "q400_one_seed_level": (150_001, 3, 768, 400, 42, True),       # ragged last query tile
    "q512_two_seed_levels": (400_037, 2, 768, 512, 43, True),
    "q1024_two_clusters_per_column": (200_003, 2, 768, 1024, 44, True),
    "single_field_q512": (300_001, 1, 768, 512, 45, True),          # two epilogue sets
    "odd_kc_dim704_q512": (100_001, 2, 704, 512, 46, False),        # 11 chunks per stage: CTA pairs only
}


@pytest.mark.parametrize("case", list(CASES))
def test_ranked_and_cluster4_path(case):
    n, F, d, Q, seed, expect_c4 = CASES[case]
    r, pc, q, w = _retriever(n, F, d, Q, seed)
    chk = Fp32Checker(pc)
    ref_s, ref_i = chk.topk(q, w, K, slack=64)
    _cluster4_ctas()
    s, i = r.search(q, q.float(), impl="tcgen05_qs")
    torch.cuda.synchronize()
    c4 = _cluster4_ctas()
    assert_topk_parity_at_scale(s, i, ref_s, ref_i, chk.rescore(q, w, i), K, n, what=case)
    if expect_c4:
        assert c4 > 0 and c4 % 4 == 0, c4
    else:
        assert c4 == 0, c4
    del r, pc, chk
    gc.collect()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("sparse_dtype", [torch.float16, torch.float32])
def test_fused_sparse_in_cluster4(sparse_dtype):
    """The fused-sparse instantiation (stages of 6 chunks, split 3 + 3) against the CPU oracle."""
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    g = torch.Generator().manual_seed(47)
    N, d, Fd, Fs, Q = 9_001, 768, 2, 2, 512
    mu = torch.randn(d, generator=g)
    fields = [O.round_bf16(torch.randn(N, d, generator=g) + 0.5 * mu) for _ in range(Fd)]
    q = O.round_bf16(torch.randn(Q, d, generator=g) + 0.5 * mu)
    sp = torch.where(torch.rand(Q, Fs, N, generator=g) < 0.95, torch.zeros(()),
                     4.0 * torch.rand(Q, Fs, N, generator=g)).half()
    W = 0.05 * torch.randn(d, Fd + Fs, generator=g)
    layer = LinearWeights(d, Fd + Fs, query_cond=True)
    with torch.no_grad():
        layer.weight.copy_(W)
    r = MultiFieldRetriever(PackedCorpus.from_fields(fields, DEV), layer.to(DEV), n_sparse=Fs, top_k=K, device=DEV)
    ref = O.exhaustive_scores(q, fields, sp.float(), O.mixture_weights(q, W, True))
    ld = (N + 63) // 64 * 64
    padded = torch.zeros((Q, Fs, ld), dtype=sparse_dtype, device=DEV)
    padded[:, :, :N] = sp.to(DEV)
    qd = q.to(DEV)
    _cluster4_ctas()
    s, i = r.search(qd, qd, padded, impl="tcgen05_qs")
    torch.cuda.synchronize()
    c4 = _cluster4_ctas()
    assert r.last_launches == 2                      # fused gather: scoring + merge
    assert_topk_parity(s.cpu().numpy(), i.cpu().numpy(), ref.numpy(), K)
    assert c4 > 0 and c4 % 4 == 0, c4
