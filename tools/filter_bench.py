"""Cost of a doc filter (``search(doc_filter=...)``, DESIGN §4.5) on one GPU: each filtered call is timed alternately
with the unfiltered call on the same corpus and queries.

    python tools/filter_bench.py --out DIR [--docs 10000000] [--steps 20] [--rounds 3]

Corpus: SYNTHETIC 10M x 8 x 768 (``mfar_b200.synth``, the generator bench.py uses), bf16 at Q in {1, 64, 512}, then the
same rows as E4M3 at Q = 64 (the two corpora do not fit together: 123 + 61 GB).  Filters: a shared all-ones row, a
shared row with half the docs eligible, a shared row with 1 %, and one row per query with half the docs eligible
(random words: every doc eligible with probability 1/2, independently).  Kernel time is what the library's CUDA
events measure around the scoring launches of a call (``mfar_profile_enable``, seeding prefix included); the report
keeps the median of each round and the median over rounds.  Writes DIR/filter_bench.json with the card's name and
power limit.
"""
from __future__ import annotations

import argparse
import ctypes
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "multifield-adaptive-retrieval_b200"))

DIM, K, SEED, F = 768, 100, 7, 8


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:                                # the numbers still stand, without the card's name
        return {"name": None, "error": str(e)}


def retriever(n, dtype, dev):
    import torch
    from mfar_b200 import synth as S
    from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
    from mfar_b200.modeling.weighting import LinearWeights
    pc = PackedCorpus(n, F, DIM, dev, dtype=dtype)
    S.fill_packed_corpus(pc, seed=SEED)
    layer = LinearWeights(DIM, F, query_cond=True)
    with torch.no_grad():
        layer.weight.copy_(S.make_mixture(DIM, F, SEED + 1))
    return MultiFieldRetriever(pc, layer.to(dev), top_k=K)


def kernel_ms(r, q, steps, warmup, doc_filter):
    """Median scoring-kernel time (ms) of `steps` calls."""
    import torch
    from mfar_b200 import _native as nv
    for _ in range(warmup):
        r.search(q, doc_filter=doc_filter)
    torch.cuda.synchronize()
    nv.check(nv.lib().mfar_profile_enable(1))
    for _ in range(steps):
        r.search(q, doc_filter=doc_filter)
    torch.cuda.synchronize()
    buf = (ctypes.c_float * 256)()
    n = nv.lib().mfar_profile_collect(buf, 256)
    nv.check(nv.lib().mfar_profile_enable(0))
    ks = sorted(buf[:n])
    return ks[len(ks) // 2]


def filters(n, batches, dev):
    import torch
    from mfar_b200.data.bm25 import safe_docs_bitmap
    W = (n + 31) // 32
    g = torch.Generator(device=dev).manual_seed(SEED)
    rng = np.random.default_rng(SEED)
    rand_words = lambda shape: torch.randint(-(1 << 31), 1 << 31, shape, generator=g, device=dev, dtype=torch.int64
                                             ).to(torch.int32)
    out = {"ones": lambda Q: shared["ones"], "shared50": lambda Q: shared["shared50"],
           "shared1": lambda Q: shared["shared1"], "per_query50": lambda Q: per_query[Q]}
    shared = {"ones": torch.from_numpy(safe_docs_bitmap(np.arange(n), n).view(np.int32)).to(dev),
              "shared50": rand_words((W,)),
              "shared1": torch.from_numpy(safe_docs_bitmap(np.flatnonzero(rng.random(n) < 0.01), n).view(np.int32)
                                          ).to(dev)}
    per_query = {Q: rand_words((Q, W)) for Q in batches}
    return out, {"shared_row_bytes": W * 4, "per_query_bytes": {Q: Q * W * 4 for Q in batches}}


def run(r, n, batches, a, dev, rep_rows, dtype):
    import torch
    from mfar_b200 import synth as S
    mu = S.corpus_mean(DIM, SEED, dev)
    qs = {Q: S.make_queries(Q, DIM, mu, SEED + 10 + Q, dev) for Q in batches}
    fl, sizes = filters(n, batches, dev)
    names = list(fl)
    t = {(Q, f): {"unfiltered": [], "filtered": []} for Q in batches for f in names}
    for _ in range(a.rounds):                             # alternate: both share the clock / power state
        for Q in batches:
            for f in names:
                t[(Q, f)]["unfiltered"].append(kernel_ms(r, qs[Q], a.steps, a.warmup, None))
                t[(Q, f)]["filtered"].append(kernel_ms(r, qs[Q], a.steps, a.warmup, fl[f](Q)))
    for Q in batches:
        for f in names:
            u, v = sorted(t[(Q, f)]["unfiltered"]), sorted(t[(Q, f)]["filtered"])
            mu_, mv = u[len(u) // 2], v[len(v) // 2]
            row = {"dtype": dtype, "Q": Q, "filter": f, "unfiltered_ms": mu_, "filtered_ms": mv,
                   "overhead_pct": 100.0 * (mv / mu_ - 1.0), "unfiltered_rounds_ms": u, "filtered_rounds_ms": v,
                   "filter_bytes": sizes["per_query_bytes"][Q] if f == "per_query50" else sizes["shared_row_bytes"],
                   "corpus_bytes": n * F * DIM * (2 if dtype == "bf16" else 1) + (n * F * 4 if dtype == "e4m3" else 0)}
            rep_rows.append(row)
            print(json.dumps({k: row[k] for k in ("dtype", "Q", "filter", "unfiltered_ms", "filtered_ms",
                                                  "overhead_pct")}), flush=True)
    del fl
    torch.cuda.synchronize()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--docs", type=int, default=10_000_000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("filter_bench needs a CUDA device (numbers are measured on the GPU only)")
    dev = torch.device("cuda:0")
    os.makedirs(a.out, exist_ok=True)
    rep = {"card": card(), "synthetic_data": True, "shape": [a.docs, F, DIM], "k": K, "steps": a.steps,
           "rounds": a.rounds, "rows": []}
    for dtype, batches in (("bf16", [1, 64, 512]), ("e4m3", [64])):
        t0 = time.time()
        r = retriever(a.docs, dtype, dev)
        torch.cuda.synchronize()
        rep[f"pack_s_{dtype}"] = time.time() - t0
        run(r, a.docs, batches, a, dev, rep["rows"], dtype)
        del r
        gc.collect()
        torch.cuda.empty_cache()
    rep["max_overhead_pct"] = max(r_["overhead_pct"] for r_ in rep["rows"])
    with open(os.path.join(a.out, "filter_bench.json"), "w") as f:
        json.dump(rep, f, indent=1)
    print(json.dumps({"card": rep["card"], "max_overhead_pct": rep["max_overhead_pct"]}), flush=True)


if __name__ == "__main__":
    main()
