#!/usr/bin/env python
"""Times the load-time corpus pack (``PackedCorpus.load_rows`` -> ``mfar_corpus_pack_rows``) of a large corpus, with or
without the cosine normalisation (needs a B200; not part of pytest).

    python tools/time_pack.py [--docs 10000000] [--fields 8] [--dim 768] [--raw] [--out pack_timing.json]

The source is one device-resident fp32 chunk of ``--chunk`` rows packed into every chunk position of every field, so
the number is the pack kernel's own time over the whole corpus (host reads and PCIe copies excluded), taken with CUDA
events around each field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_p = os.path.join(ROOT, "multifield-adaptive-retrieval_b200")
if _p not in sys.path:
    sys.path.insert(0, _p)

import torch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--docs", type=int, default=10_000_000)
    ap.add_argument("--fields", type=int, default=8)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--chunk", type=int, default=131072)
    ap.add_argument("--raw", action="store_true", help="pack without normalisation")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    from mfar_b200.modeling.retrieval import PackedCorpus
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    src = torch.randn(a.chunk, a.dim, generator=g, device=dev) * 3 + 0.5
    pc = PackedCorpus(a.docs, a.fields, a.dim, dev, normalize=not a.raw)
    pc.load_rows(0, 0, src[:1000])                          # module load, launch attributes
    torch.cuda.synchronize()
    per_field = []
    for f in range(a.fields):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for lo in range(0, a.docs, a.chunk):
            pc.load_rows(f, lo, src[:min(a.chunk, a.docs - lo)])
        ev[1].record()
        torch.cuda.synchronize()
        per_field.append(ev[0].elapsed_time(ev[1]))
    total_ms = sum(per_field)
    elems = a.docs * a.fields * a.dim
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                          "0"], capture_output=True, text=True).stdout.strip()
    res = dict(docs=a.docs, fields=a.fields, dim=a.dim, normalize=not a.raw, chunk=a.chunk, total_ms=round(total_ms, 2),
               field_ms=[round(x, 2) for x in per_field],
               gb_per_s=round(elems * (4 + 2) / (total_ms * 1e-3) / 1e9, 1), gpu=smi)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
