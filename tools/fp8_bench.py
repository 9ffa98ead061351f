"""bf16 vs E4M3 corpus on one GPU: scoring-kernel time, bytes/s and FLOP/s against the B200 data sheet, which bound
each shape sits at, and how far the E4M3 top-100 moves from the bf16 top-100.  Then the 20M x 8 x 768 E4M3 corpus
(245 GB in bf16) on one GPU, with a sample of its answers re-scored by ``score_candidates``.

    python tools/fp8_bench.py --out DIR [--docs 10000000] [--big-docs 20000000] [--steps 20] [--rounds 3]

The corpora and queries are SYNTHETIC (``mfar_b200.synth``: Gaussian rows around a shared mean, the generator bench.py
uses), so the top-100 overlap says how E4M3 rounding reorders near neighbours of such data, not what it does to a
trained encoder's embeddings.  Both corpora are packed from the same fp32 rows.  bf16 and E4M3 are timed alternately
in the same process, each call's kernel time from the library's CUDA events (``mfar_profile_enable``: the scoring
launches of a call, seeding prefix included).  Writes DIR/fp8_bench.json.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "multifield-adaptive-retrieval_b200"))

HBM_BPS = 7.7e12            # B200 data sheet, one GPU
PEAK = {"bf16": 2.25e15, "e4m3": 4.5e15}   # dense tensor FLOP/s, B200 data sheet (for a card allowed 1,000 W)
DIM, K, SEED = 768, 100, 7


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:                                # the numbers still stand, without the card's name
        return {"name": None, "error": str(e)}


def build(n, F, dtype, dev):
    from mfar_b200 import synth as S
    from mfar_b200.modeling.retrieval import PackedCorpus
    pc = PackedCorpus(n, F, DIM, dev, dtype=dtype)
    S.fill_packed_corpus(pc, seed=SEED)
    return pc


def retriever(pc, F, dev):
    import torch
    from mfar_b200 import synth as S
    from mfar_b200.modeling.retrieval import MultiFieldRetriever
    from mfar_b200.modeling.weighting import LinearWeights
    layer = LinearWeights(DIM, F, query_cond=True)
    with torch.no_grad():
        layer.weight.copy_(S.make_mixture(DIM, F, SEED + 1))
    return MultiFieldRetriever(pc, layer.to(dev), top_k=K)


def time_calls(r, q, steps, warmup):
    """Median per-call scoring-kernel time (ms) and the mean wall time of a call ending in a synchronise."""
    import torch
    from mfar_b200 import _native as nv
    for _ in range(warmup):
        r.search(q)
    torch.cuda.synchronize()
    nv.check(nv.lib().mfar_profile_enable(1))
    t0 = time.perf_counter()
    for _ in range(steps):
        r.search(q)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / steps * 1e3
    import ctypes
    buf = (ctypes.c_float * 256)()
    n = nv.lib().mfar_profile_collect(buf, 256)
    nv.check(nv.lib().mfar_profile_enable(0))
    ks = sorted(buf[:n])
    return ks[len(ks) // 2], wall


def roofline(n, F, Q, dtype, kernel_ms):
    elem = 2 if dtype == "bf16" else 1
    bytes_ = n * F * DIM * elem + (n * F * 4 if dtype == "e4m3" else 0)
    flops = 2.0 * Q * n * F * DIM
    t_bw, t_fl = bytes_ / HBM_BPS, flops / PEAK[dtype]
    s = kernel_ms / 1e3
    return {"bytes": bytes_, "flops": flops, "bytes_per_s": bytes_ / s, "flop_per_s": flops / s,
            "hbm_share": bytes_ / s / HBM_BPS, "tensor_share": flops / s / PEAK[dtype],
            "bound": "HBM" if t_bw >= t_fl else "tensor", "share_of_bound": max(t_bw, t_fl) / s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--docs", type=int, default=10_000_000)
    ap.add_argument("--fields", type=int, default=8)
    ap.add_argument("--big-docs", type=int, default=20_000_000)
    ap.add_argument("--batches", default="1,64,512")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import torch
    from mfar_b200 import synth as S
    if not torch.cuda.is_available():
        sys.exit("fp8_bench needs a CUDA device (numbers are measured on the GPU only)")
    dev = torch.device("cuda:0")
    os.makedirs(a.out, exist_ok=True)
    F, batches = a.fields, [int(x) for x in a.batches.split(",")]
    rep = {"card": card(), "synthetic_data": True, "shape": [a.docs, F, DIM], "k": K,
           "peaks": {"hbm_bytes_per_s": HBM_BPS, "dense_flop_per_s": PEAK}}
    free = torch.cuda.mem_get_info()[0]
    need = a.docs * F * DIM * 3 + a.docs * F * 4 + 4e9
    n = a.docs if free >= need else int((free - 4e9) / (F * (DIM * 3 + 4))) // 128 * 128
    rep["docs_timed"] = n
    rep["note_docs"] = "" if n == a.docs else f"both corpora resident needs {need / 1e9:.0f} GB; ran {n} docs"
    t0 = time.time()
    rs = {d: retriever(build(n, F, d, dev), F, dev) for d in ("bf16", "e4m3")}
    torch.cuda.synchronize()
    rep["pack_s"] = time.time() - t0
    mu = S.corpus_mean(DIM, SEED, dev)
    qs = {Q: S.make_queries(Q, DIM, mu, SEED + 10 + Q, dev) for Q in batches}
    runs = {(d, Q): [] for d in rs for Q in batches}
    for _ in range(a.rounds):                              # alternate: bf16 and E4M3 share the clock / power state
        for Q in batches:
            for d in ("bf16", "e4m3"):
                runs[(d, Q)].append(time_calls(rs[d], qs[Q], a.steps, a.warmup))
    rep["shapes"] = []
    for Q in batches:
        row = {"Q": Q}
        for d in ("bf16", "e4m3"):
            ks = sorted(x[0] for x in runs[(d, Q)])
            row[d] = {"kernel_ms": ks[len(ks) // 2], "kernel_ms_all_rounds": ks,
                      "call_ms": min(x[1] for x in runs[(d, Q)]), **roofline(n, F, Q, d, ks[len(ks) // 2])}
        row["speedup"] = row["bf16"]["kernel_ms"] / row["e4m3"]["kernel_ms"]
        _, ib = rs["bf16"].search(qs[Q])
        _, ie = rs["e4m3"].search(qs[Q])
        ov = [len(set(ib[j].tolist()) & set(ie[j].tolist())) / K for j in range(Q)]
        row["top100_overlap_mean"], row["top100_overlap_min"] = sum(ov) / Q, min(ov)
        rep["shapes"].append(row)
        print(json.dumps({k: row[k] for k in ("Q", "speedup", "top100_overlap_mean")}
                         | {d: row[d]["kernel_ms"] for d in ("bf16", "e4m3")}), flush=True)
    del rs
    gc.collect()
    torch.cuda.empty_cache()

    # ---- the corpus that needs two GPUs in bf16, on one in E4M3
    nb = a.big_docs
    big = {"shape": [nb, F, DIM], "bf16_bytes": nb * F * DIM * 2, "e4m3_bytes": nb * F * DIM + nb * F * 4}
    free = torch.cuda.mem_get_info()[0]
    big["free_hbm_bytes"] = free
    if free < big["e4m3_bytes"] + 4e9:
        big["skipped"] = "does not fit"
    else:
        t0 = time.time()
        r = retriever(build(nb, F, "e4m3", dev), F, dev)
        torch.cuda.synchronize()
        big["pack_s"] = time.time() - t0
        q = qs[64]
        km, wall = time_calls(r, q, a.steps, a.warmup)
        big["Q64"] = {"kernel_ms": km, "call_ms": wall, **roofline(nb, F, 64, "e4m3", km)}
        s, i = r.search(q)
        m = 8                                              # a sample of the answers, re-scored field by field
        per_field = r.score_candidates(q[:m], i[:m].reshape(-1))               # [F, m, m*K]
        w = r.mixture.field_weights(r.mixture_input(q[:m]), r.mask, batch=m)   # [m, F]
        mixed = torch.einsum("fqc,qf->qc", per_field, w).view(m, m, K)
        resc = torch.stack([mixed[j, j] for j in range(m)])
        err = ((resc - s[:m]).abs() / s[:m].abs().clamp(min=1e-6)).max().item()
        big["sample_rescore_max_rel_err"] = err
        big["sample_queries"] = m
        big["sample_sorted"] = bool((s[:, 1:] <= s[:, :-1]).all().item())
        del r
    rep["big"] = big
    with open(os.path.join(a.out, "fp8_bench.json"), "w") as f:
        json.dump(rep, f, indent=1)
    print(json.dumps({"card": rep["card"], "big": {k: v for k, v in big.items() if k != "Q64"}}), flush=True)


if __name__ == "__main__":
    main()
