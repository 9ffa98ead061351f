#!/usr/bin/env python
"""bench.py - queries/sec of exhaustive multi-field top-100 on synthetic STaRK-shaped corpora.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload scale_10m_all] [--batch 512] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's CPU pipeline on the host cores

One "step" = one batch of Q queries scored against the whole corpus (all fields), mixed, top-100.
Multi-GPU = strong scaling: the SAME global corpus is doc-range sharded over the ranks, per-shard top-k keys are
exchanged and merged by one kernel over NVLink peer memory (NCCL all-gather + merge kernel as fallback).
Rank 0 prints ONE JSON line: the headline workload (BASELINE.json configs[4], batch 512) with `roofline`,
`cpu_baseline`, `e2e`, `parity_check`, `other_batches` (batch 1 / 64 of the same corpus, at every N) and
`other_workloads` (C2 PRIME hybrid, C3 MAG, C4 Amazon hybrid, C5 single_), each with its own roofline and parity check.
"""
from __future__ import annotations

import argparse
import ctypes
import gc
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.join(ROOT, "multifield-adaptive-retrieval_b200"), os.path.join(ROOT, "oracle"),
           os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

METRIC = "queries/sec for multi-field top-100"
NOMINAL_HBM_GBS = 8000.0        # north_star: "roughly 8 TB/s" (BASELINE.md section 2: fractions against both, labelled)
NOMINAL_BF16_TFLOPS = 2250.0    # dense bf16, B200 data sheet
DIM = 768
TOPK = 100
GEN_CHUNK = 65536
DUMP_BYTES = 64_000_000         # --dump-outputs: at most this much in all
# what rides along with the headline in the default run: (workload, batches) - BASELINE.json configs 2, 3, 4 and the
# single_ scorer of config 5
OTHER_WORKLOADS = (("prime_full", (1, 64)), ("mag_full", (1, 512)), ("amazon_full", (64, 512)),
                   ("scale_10m_single", (1, 64, 512)))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ---------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            c = [x.strip() for x in r.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def algorithmic_work(n_docs, n_dense, n_sparse, Q, sparse_bytes=2):
    """BASELINE.md section 3: bytes = N*Fd*d*2 (+ Q*N*Fs*b_s) + small; flops = 2*Q*N*Fd*d."""
    bytes_ = n_docs * n_dense * DIM * 2 + Q * n_docs * n_sparse * sparse_bytes + Q * DIM * 2 + Q * TOPK * 12
    flops = 2.0 * Q * n_docs * n_dense * DIM
    return bytes_, flops


# ---------------------------------------------------------------------------------------- CPU arm
def cpu_reference_leg(n_total, n_dense, n_sparse, Q, seed, steps, warmup):
    """The reference's CPU pipeline (``trec_eval_step``: per-field retrieve_batch -> union -> per-query score_batch ->
    mask -> mixture -> top-100) on all host threads, on a FIXED bounded sample: 200,000 docs (or the corpus, if smaller)
    and min(Q, 64) queries - 64 is the reference's own dev batch.  Driven through oracle/cpu_pipeline.py: the reference's
    own DenseFlatIndex / MemoryMapDict / LinearWeights when /root/reference is present (kind "reference"), else the
    port that pays the same per-call costs (kind "port").  The per-step time is linear in the doc count with a
    per-query constant (the union / rescore / Python part): t(n) = a + b*n is fitted from a second, 50,000-doc sample
    and ONLY the fitted line is evaluated at the full size - value = Q_s / (a + b*n_total)."""
    import cpu_pipeline as C
    import ref_import
    torch.set_num_threads(os.cpu_count() or 1)
    kind = "reference" if ref_import.available() else "port"
    q_s = min(Q, 64)
    n2 = min(n_total, 200_000)
    n1 = min(n_total, 50_000)
    make_rows = None
    if torch.cuda.is_available():                     # draw the sample on the GPU (setup only; everything timed is CPU)
        g = torch.Generator(device="cuda").manual_seed(seed)
        mu = torch.randn(DIM, generator=g, device="cuda")

        def make_rows(n, d, f):
            return (torch.randn(n, d, generator=g, device="cuda") + 0.5 * mu).to(torch.bfloat16).float().cpu().numpy()
    tmp_root = None                                   # field memmaps: tmpfs when there is room (the reference's temp_dir
    try:                                              # is served from the page cache once touched), else the default
        st = os.statvfs("/dev/shm")
        if st.f_bavail * st.f_frsize > 2 * n2 * max(n_dense, 1) * DIM * 4:
            tmp_root = "/dev/shm"
    except OSError:
        pass
    t2 = C.time_pipeline(kind, n2, n_dense, n_sparse, q_s, DIM, seed, steps=steps, warmup=warmup, make_rows=make_rows,
                         tmp_root=tmp_root)
    t_step = statistics.median(t2)
    if n1 < n2:
        t1 = statistics.median(C.time_pipeline(kind, n1, n_dense, n_sparse, q_s, DIM, seed, steps=3, warmup=1,
                                               make_rows=make_rows, tmp_root=tmp_root))
        b = max((t_step - t1) / (n2 - n1), 0.0)
        a = max(t_step - b * n2, 0.0)
        t_full = a + b * n_total
    else:
        a, b, t_full = t_step, 0.0, t_step
    extrap = n_total > n2
    sample = (f"{kind} of trec_eval_step (oracle/cpu_pipeline.py), fp32 torch/numpy on {torch.get_num_threads()} host "
              f"threads, field memmaps on disk; timed on {n2} of {n_total} docs x {n_dense}+{n_sparse} fields, "
              f"{q_s} queries per step, median of {steps}"
              + (f"; t(n) = a + b*n fitted with a {n1}-doc sample and evaluated at {n_total} docs" if extrap else ""))
    return {"value": q_s / t_full, "unit": "queries/s", "cores": torch.get_num_threads(), "kind": kind, "sample": sample,
            "ms_per_step_sample": t_step * 1e3, "n_sample": n2, "queries_per_step": q_s,
            "fit_a_s": a, "fit_b_s_per_doc": b, "extrapolated": extrap, "os_cpu_count": os.cpu_count(),
            "cpu_model": cpu_model()}


# ---------------------------------------------------------------------------------------- GPU arm
class Ctx:
    """Process-wide state of our arm: device, ranks, the peer exchange, shard weights."""

    def __init__(self, args):
        import torch.distributed as dist
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        self.dist = dist
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.device)
        self.exchange, self.exchange_kind = None, "none (1 GPU)"
        if self.world > 1:
            from mfar_b200.dist import PeerExchange
            if os.environ.get("MFAR_EXCHANGE", "p2p") == "p2p":
                try:
                    self.exchange = PeerExchange(q_cap=max(1024, args.batch), k_cap=128, device=self.device)
                    self.exchange_kind = "fused NVLink peer-memory exchange+merge kernel (mfar_topk_exchange_merge)"
                except Exception as e:  # noqa: BLE001  (symmetric memory unavailable: NCCL all-gather + merge kernel)
                    self.exchange_kind = (f"nccl all_gather + merge kernel (peer exchange unavailable: "
                                          f"{type(e).__name__}: {e})")[:300]
            else:
                self.exchange_kind = "nccl all_gather + merge kernel"
        self.peaks = load_peaks()
        self.pipelined = self.exchange is not None and args.exchange_mode == "pipelined"
        self.weights = [1.0] * self.world             # relative docs/s of every rank (calibrated when --balance)
        self.balance_note = "equal doc ranges"

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = torch.tensor([x], device=self.device, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def per_rank(self, x: float):
        if self.world == 1:
            return [x]
        t = torch.zeros(self.world, device=self.device, dtype=torch.float64)
        t[self.rank] = x
        self.dist.all_reduce(t)
        return t.tolist()

    def calibrate(self, n_dense, Q, shard_docs, seconds=1.5):
        """Speed-weighted shards: the job runs at the pace of its slowest rank, and the GPUs of a node settle at different
        clocks under the 1 kW cap (a few per cent apart).  Each rank times the scoring kernel on an identical calibration
        shard of the REAL shard size (so the kernel is in the same power-capped regime as in the run; capped at 2.5M docs)
        for `seconds` of sustained load; doc ranges are then sized in proportion to the measured docs/s."""
        from mfar_b200 import synth
        from mfar_b200.modeling.retrieval import MultiFieldRetriever, PackedCorpus
        from mfar_b200.modeling.weighting import LinearWeights
        n = int(min(max(shard_docs, 131072), 2_500_000))
        pc = PackedCorpus(n, max(n_dense, 1), DIM, self.device)
        synth.fill_packed_corpus(pc, seed=99)
        mu = synth.corpus_mean(DIM, 99, self.device)
        layer = LinearWeights(DIM, max(n_dense, 1), query_cond=True).to(self.device)
        r = MultiFieldRetriever(pc, layer, top_k=TOPK)
        q = synth.make_queries(Q, DIM, mu, 98, self.device)
        qe = q.float()
        for _ in range(3):
            r.search(q, qe)
        self.barrier()
        t_end = time.perf_counter() + seconds
        laps = []
        while time.perf_counter() < t_end:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                r.search(q, qe)
            e1.record()
            e1.synchronize()
            laps.append(e0.elapsed_time(e1) / 10)
        mine = statistics.median(laps[len(laps) // 2:])          # the settled second half
        t = torch.zeros(self.world, device=self.device, dtype=torch.float64)
        t[self.rank] = mine
        self.dist.all_reduce(t)
        ms = t.tolist()
        self.weights = [1.0 / max(x, 1e-9) for x in ms]
        spread = (max(ms) - min(ms)) / min(ms)
        self.balance_note = (f"speed-weighted doc ranges (calibration kernel ms per rank: "
                             f"{', '.join(f'{x:.3f}' for x in ms)}; spread {100 * spread:.1f} %)")
        del r, pc
        torch.cuda.empty_cache()


def build_shard(n_total, n_fields, lo, hi, seed, device):
    """Rank-local PackedCorpus holding global docs [lo, hi).  Generation is per global 64k-doc chunk so every
    shard count (and every shard boundary) sees the same global corpus."""
    from mfar_b200 import synth
    from mfar_b200.modeling.retrieval import PackedCorpus
    pc = PackedCorpus(hi - lo, n_fields, DIM, device)
    mu = synth.corpus_mean(DIM, seed, device)
    c0, c1 = lo // GEN_CHUNK, (hi - 1) // GEN_CHUNK
    for c in range(c0, c1 + 1):
        g = torch.Generator(device=device)
        g.manual_seed(seed * 1000003 + c + 1)
        clo, chi = c * GEN_CHUNK, min(n_total, (c + 1) * GEN_CHUNK)
        a, b = max(lo, clo), min(hi, chi)
        for f in range(n_fields):
            rows = synth.make_field_rows(chi - clo, DIM, mu, g, device)
            pc.load_rows(f, a - lo, rows[a - clo:b - clo])
    torch.cuda.synchronize()
    return pc, mu


class Workload:
    """One corpus (this rank's shard of it), its retriever, and the timing / checking legs."""

    def __init__(self, ctx: Ctx, name: str, docs_override: int = 0):
        from mfar_b200 import synth
        from mfar_b200.dist import ShardedRetriever, held_ranges, weighted_shard_ranges
        from mfar_b200.modeling.weighting import LinearWeights
        self.ctx, self.name = ctx, name
        a = ctx.args
        self.n_total, self.n_dense, self.n_sparse = synth.SHAPES[name]
        if docs_override:
            self.n_total = docs_override
        self.bm25_mode = a.sparse_mode == "bm25" and self.n_sparse > 0
        ranges = weighted_shard_ranges(self.n_total, ctx.weights)
        self.cuts = self.base_cuts = [r[0] for r in ranges] + [self.n_total]
        self.lo, self.hi = ranges[ctx.rank]
        # Tunable boundaries (dense-only scorers at N > 1, --balance auto): every rank keeps a margin of its neighbours'
        # docs resident, so the boundaries can follow the measured per-rank step time (tune_boundaries) by pointer offset.
        self.margin = 0
        if ctx.world > 1 and a.balance == "auto" and self.n_dense and not self.n_sparse:
            self.margin = -(-int(0.06 * self.n_total / ctx.world) // 128) * 128
        self.held_lo, self.held_hi = held_ranges(self.cuts, self.margin, self.n_total)[ctx.rank]
        self.tuning = None
        t0 = time.perf_counter()
        if self.n_dense:
            self.pc_held, self.mu = build_shard(self.n_total, self.n_dense, self.held_lo, self.held_hi, a.seed,
                                                ctx.device)
            self.pc = self.pc_held if not self.margin else self.pc_held.window(self.lo - self.held_lo, self.hi - self.lo)
        else:                                             # sparse-only scorer: nothing to pack
            self.pc_held = self.pc = None
            self.mu = synth.corpus_mean(DIM, a.seed, ctx.device)
        F = self.n_dense + self.n_sparse
        layer = LinearWeights(DIM, F, query_cond=True)
        with torch.no_grad():
            layer.weight.copy_(synth.make_mixture(DIM, F, a.seed + 1))
        self.layer = layer.to(ctx.device)
        self.bm25_fields = None
        if self.bm25_mode:
            self.bm25_fields = [synth.make_bm25_field(self.n_total, a.seed + 300 + j, ctx.device,
                                                      doc_range=(self.lo, self.hi)) for j in range(self.n_sparse)]
            torch.cuda.synchronize()
        self.graphs = {}
        self._make_retriever()
        self.setup_s = time.perf_counter() - t0

    def _make_retriever(self):
        from mfar_b200.dist import ShardedRetriever
        from mfar_b200.modeling.retrieval import MultiFieldRetriever
        ctx, a = self.ctx, self.ctx.args
        self.graphs.clear()
        self.retr = MultiFieldRetriever(self.pc, self.layer, n_sparse=self.n_sparse, top_k=TOPK, doc_id_base=self.lo,
                                        impl=a.kernel, sparse_indices=self.bm25_fields, n_docs=self.hi - self.lo,
                                        device=ctx.device)
        self.sharded = ShardedRetriever(self.retr, exchange=ctx.exchange)               # complete exchange per call
        # throughput mode of the timed loops: a step pushes its keys and merges the PREVIOUS step's, so no rank waits
        # for the slowest rank of the current step (results trail by one step; flush() returns the last one)
        self.piped = ShardedRetriever(self.retr, exchange=ctx.exchange, pipelined=ctx.pipelined)

    def tune_boundaries(self, Q, rounds=4, steps=10, tol=0.006):
        """Start-up, untimed: run the real sharded step, measure every rank's scoring-kernel time, move the shard
        boundaries towards equal time (dist.rebalanced_boundaries), repeat.  Stops when the spread over the ranks is
        below `tol`.  The history goes into the JSON line (config.sharding)."""
        from mfar_b200 import _native as nv
        from mfar_b200.dist import rebalanced_boundaries
        ctx = self.ctx
        if not self.margin:
            return
        pool = self.make_batches(Q, 2)
        hist = []
        for it in range(rounds + 1):
            for i in range(3):
                self.step(pool[i % 2], False)
            ctx.barrier()
            nv.check(nv.lib().mfar_profile_enable(1))
            for i in range(steps):
                self.step(pool[i % 2], False)
            ctx.barrier()
            km = self._collect_profile()
            ts = ctx.per_rank(statistics.mean(km) if km else 0.0)
            spread = (max(ts) - min(ts)) / max(min(ts), 1e-9)
            hist.append({"kernel_ms": [round(x, 4) for x in ts], "spread": round(spread, 4),
                         "cuts_minus_equal": [c - b for c, b in zip(self.cuts, self.base_cuts)]})
            if spread < tol or it == rounds:
                break
            self.cuts = rebalanced_boundaries(self.cuts, ts, self.base_cuts, self.margin)
            self.lo, self.hi = self.cuts[ctx.rank], self.cuts[ctx.rank + 1]
            self.pc = self.pc_held.window(self.lo - self.held_lo, self.hi - self.lo)
            self._make_retriever()
        self.tuning = hist
        del pool

    # ------------------------------------------------------------------ inputs
    def make_batches(self, Q, n_pool=4):
        from mfar_b200 import synth
        a, dev = self.ctx.args, self.ctx.device
        n_shard = self.hi - self.lo
        if self.n_sparse and not self.bm25_mode:          # keep the pool of [Q,Fs,N] f16 tensors within a few GB
            n_pool = max(1, min(n_pool, int(6e9 // max(1, Q * self.n_sparse * n_shard * 2))))
        pool = []
        for i in range(n_pool):
            qv = synth.make_queries(Q, DIM, self.mu, a.seed + 100 + i, dev)
            sp = ent = None
            if self.bm25_mode:
                ent = synth.make_bm25_query_entries(Q, self.n_sparse, a.seed + 200 + i).to(dev)
            elif self.n_sparse:
                ld = (n_shard + 63) // 64 * 64            # 128-byte row pitch: gathered inside the scoring epilogue
                sp = torch.zeros((Q, self.n_sparse, ld), dtype=torch.float16, device=dev)
                for q0 in range(0, Q, 32):                # shard columns [lo, hi) of the global sparse tensor
                    q1 = min(Q, q0 + 32)
                    full = synth.make_sparse(q1 - q0, self.n_sparse, self.n_total, a.seed + 200 + 1000 * i + q0, dev)
                    sp[q0:q1, :, :n_shard] = full[:, :, self.lo:self.hi]
                    del full
            pool.append((qv, qv.float(), sp, ent))
        return pool

    # ------------------------------------------------------------------ one step
    def step(self, batch, graph: bool):
        qv, qe, sp, ent = batch
        if graph:
            key = (qv.shape[0], 0 if sp is None else sp.data_ptr())      # one graph per resident sparse tensor
            gs = self.graphs.get(key)
            if gs is None:
                from mfar_b200.modeling.retrieval import GraphedSearch
                gs = self.graphs[key] = GraphedSearch(
                    self.retr, qv.shape[0], sparse="bm25" if self.bm25_mode else ("dense" if self.n_sparse else "none"),
                    max_entries=0 if ent is None else ent.shape[0], sparse_buffer=sp,
                    sharded=self.piped if self.ctx.world > 1 else None)
            out = gs(qv, qe, sparse=sp, entries=ent)
            return out, gs.launches
        out = self.piped.search(qv, qe, sp, sparse_tokens=ent) if self.ctx.world > 1 else \
            self.retr.search(qv, qe, sp, sparse_tokens=ent)
        extra = 1 + (0 if self.ctx.world == 1 else (1 if self.ctx.exchange is None else (3 if self.piped.pipelined else 2)))
        return out, self.retr.last_launches + extra       # + mixture weights (+ epoch bump + exchange kernels / merge)

    def time_device(self, pool, steps, warmup, graph: bool, profile: bool, sample_clocks=False, keep_last=False):
        """K timed steps with device-resident inputs.  Returns (ms total [max over ranks], launches, kernel ms list,
        clocks).  The scoring kernel's own duration comes from the library's CUDA-event pair around it; a graph replay
        carries no such events, so with `graph` the kernel is timed in a separate eager pass of the same length.
        With `keep_last`, the (scores, ids) the last timed step returned are copied to the host as `last_outputs`
        before anything else runs (a graph replay returns static buffers that later steps overwrite)."""
        from mfar_b200 import _native as nv
        ctx = self.ctx
        for i in range(warmup):
            self.step(pool[i % len(pool)], graph)
        ctx.barrier()
        sampler = ClockSampler(ctx.local_rank) if (sample_clocks and ctx.rank == 0) else None
        if sampler:
            sampler.start()
        prof = profile and not graph
        if prof:
            nv.check(nv.lib().mfar_profile_enable(1))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches = 0
        ncu_range = os.environ.get("MFAR_NCU_RANGE") == "1"      # ncu --profile-from-start off: timed regions only
        if ncu_range:
            torch.cuda.profiler.start()
        e0.record()
        for i in range(steps):
            out, n = self.step(pool[i % len(pool)], graph)
            launches += n
        e1.record()
        ctx.barrier()
        if ncu_range:
            torch.cuda.profiler.stop()
        if keep_last:
            self.last_outputs = tuple(t.cpu() for t in out)
        ms_local = e0.elapsed_time(e1)
        ms = ctx.max_over_ranks(ms_local)
        self.last_per_rank_ms_per_step = [x / steps for x in ctx.per_rank(ms_local)]
        clocks = sampler.stop() if sampler else None
        kern_ms = []
        if prof:
            kern_ms = self._collect_profile()
        elif profile:                                      # graph: eager pass for the kernel's own duration
            for i in range(min(warmup, 3)):
                self.step(pool[i % len(pool)], False)
            ctx.barrier()
            nv.check(nv.lib().mfar_profile_enable(1))
            for i in range(steps):
                self.step(pool[i % len(pool)], False)
            ctx.barrier()
            kern_ms = self._collect_profile()
        self.last_per_rank_kernel_ms = ctx.per_rank(statistics.mean(kern_ms) if kern_ms else 0.0)
        return ms, launches, kern_ms, clocks

    @staticmethod
    def _collect_profile():
        from mfar_b200 import _native as nv
        buf = (ctypes.c_float * 256)()
        n = nv.lib().mfar_profile_collect(ctypes.addressof(buf), 256)
        nv.lib().mfar_profile_enable(0)
        return [buf[i] for i in range(max(n, 0))]

    def time_e2e(self, pool, steps, warmup, graph: bool):
        """Host buffers in, host result out, every step.  N=1: ONE C-ABI call (mfar_search_host: H2D of the batch,
        mixture weights, scoring, top-k, D2H, stream sync).  N>1: pinned host -> device copies, the sharded step
        (graph replay), D2H of the merged [Q,100] result."""
        ctx = self.ctx
        n_shard = self.hi - self.lo
        pool_host = [(qv.cpu().pin_memory(), qe.cpu().pin_memory(),
                      None if sp is None else sp[:, :, :n_shard].contiguous().cpu().pin_memory(),
                      None if ent is None else ent.cpu().pin_memory()) for qv, qe, sp, ent in pool[:2]]
        Q = pool[0][0].shape[0]
        out_s = torch.empty((Q, TOPK), dtype=torch.float32).pin_memory()
        out_i = torch.empty((Q, TOPK), dtype=torch.int64).pin_memory()
        dev_sp = None if pool[0][2] is None else torch.zeros_like(pool[0][2])

        def one(i):
            qh, qeh, sph, enth = pool_host[i % len(pool_host)]
            if ctx.world == 1:
                if self.bm25_mode:
                    self.retr.search_host_bm25(qh, qeh, enth, out_scores=out_s, out_ids=out_i)
                else:
                    self.retr.search_host(qh, qeh, sph, out_scores=out_s, out_ids=out_i)
                return
            qv = qh.to(ctx.device, non_blocking=True)
            qe = qeh.to(ctx.device, non_blocking=True)
            if sph is not None:
                dev_sp[:, :, :n_shard].copy_(sph, non_blocking=True)
            ent = None if enth is None else enth.to(ctx.device, non_blocking=True)
            (s, ids), _ = self.step((qv, qe, dev_sp, ent), graph)
            out_s.copy_(s, non_blocking=True)
            out_i.copy_(ids, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        for i in range(warmup):
            one(i)
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            one(i)
        e1.record()
        ctx.barrier()
        ms = ctx.max_over_ranks(e0.elapsed_time(e1))
        if self.bm25_mode:
            h2d = Q * DIM * 2 + Q * DIM * 4 + pool[0][3].shape[0] * 12
        else:
            h2d = Q * DIM * 2 + Q * DIM * 4 + (Q * self.n_sparse * n_shard * 2 if self.n_sparse else 0)
        return ms, h2d, Q * TOPK * 12

    # ------------------------------------------------------------------ roofline of the scoring kernel
    def roofline(self, Q, k_ms, n_kernels, ms_total, steps):
        """Per launch, this rank's shard.  The fused scoring kernel moves the corpus AND (dense-tensor input, gathered in
        its epilogue) the sparse rows; with device BM25 the postings are moved by the scatter kernel, and the scoring
        kernel reads the fp32 base block instead."""
        a, peaks = self.ctx.args, self.ctx.peaks
        n_shard = self.hi - self.lo
        if k_ms is None:
            return None
        if self.n_dense == 0:
            a_bytes, a_flops = Q * n_shard * 4 + Q * TOPK * 12, 0.0            # streaming top-k of the fp32 rows
            kname = "topk_rows_kernel"
        else:
            a_bytes, a_flops = algorithmic_work(n_shard, self.n_dense, 0 if self.bm25_mode else self.n_sparse, Q)
            if self.bm25_mode:
                a_bytes += Q * n_shard * 4                                      # base[Q,N] read by the epilogue
            kname = {"simt": "score_simt_kernel", "tcgen05": "score_tc_kernel", "tcgen05_qs": "score_qs_kernel"}.get(
                a.kernel, "score_qs_kernel" if Q > 64 else "score_tc_kernel")
        hbm_bound = Q < 200 or self.n_dense == 0
        if hbm_bound:
            achieved = a_bytes / (k_ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": achieved / peaks["hbm_gbs"], "frac_of_nominal_peak": achieved / NOMINAL_HBM_GBS,
                    "nominal_peak": NOMINAL_HBM_GBS}
        else:
            achieved = a_flops / (k_ms * 1e-3) / 1e12
            roof = {"bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                    "frac": achieved / peaks["bf16_tflops_sustained"],
                    "frac_of_burst_peak": achieved / peaks["bf16_tflops"],
                    "frac_of_nominal_peak": achieved / NOMINAL_BF16_TFLOPS, "nominal_peak": NOMINAL_BF16_TFLOPS,
                    "hbm_gbs_same_launch": a_bytes / (k_ms * 1e-3) / 1e9}
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath) and self.ctx.world == 1 and not a.docs:
            traffic = json.load(open(tpath)).get(f"{self.name}|{Q}")
        roof.update({"traffic": traffic,
                     "traffic_source": "ncu --set full capture of this kernel at this shape, profiles/ncu_traffic.json "
                                       "(a profiler pass, not re-measured in this run)" if traffic else None,
                     "kernel": kname, "kernel_ms": k_ms,
                     "kernel_ms_is": "mean CUDA-event time, on the launch stream, around ALL scoring launches of a call: "
                                     "the main pass and, where threshold seeding applies (Q >= 32, >= 16 tiles per CTA), "
                                     "its one or two prefix passes of the same kernel with their merge / seed kernels in "
                                     "between - together they read the corpus once (the algorithmic bytes / flops below)",
                     "kernel_share_of_step": k_ms * steps / ms_total if ms_total else None,
                     "algorithmic_bytes_per_launch": a_bytes, "algorithmic_flops_per_launch": a_flops,
                     "peak_source": peaks["source"] + (" copy bandwidth" if hbm_bound else
                                                       " (sustained: kernel timed inside a long step)")})
        return roof

    # ------------------------------------------------------------------ what was timed is also checked
    def parity_check(self, batch, n_check=4):
        """(1) N>1: the fused NVLink exchange+merge result of the batch equals, bit for bit, the NCCL path (all-gather
        of the per-shard keys + mfar_topk_merge).  (2) the first `n_check` queries are ranked against tests/checker.py
        (plain torch fp32 over the packed corpus, TF32 off, each rank its shard, candidates all-gathered) with the
        near-tie rule of tests/parity.py - a dropped winner fails."""
        from checker import Fp32Checker, assert_topk_parity_at_scale
        from mfar_b200.dist import all_gather_keys, merge_keys
        ctx = self.ctx
        qv, qe, sp, ent = batch
        res = {"queries": 0, "ok": False}
        try:
            if ctx.world > 1:
                s, ids = self.sharded.search(qv, qe, sp, sparse_tokens=ent)
            else:
                s, ids = self.retr.search(qv, qe, sp, sparse_tokens=ent)
            if ctx.world > 1:
                _, _, keys = self.retr.search(qv, qe, sp, return_keys=True, sparse_tokens=ent)
                s2, i2 = merge_keys(all_gather_keys(keys), TOPK)
                same = bool(torch.equal(s, s2) and torch.equal(ids, i2))
                res["fused_exchange_equals_nccl_path"] = same
                if not same:
                    raise AssertionError("fused exchange result differs from all_gather + merge")
                if self.piped.pipelined:                  # the pipelined exchange delivers the same lists, one call later
                    self.piped.search(qv, qe, sp, sparse_tokens=ent)
                    s3, i3 = self.piped.search(qv, qe, sp, sparse_tokens=ent)          # = result of the first call
                    s4, i4 = self.piped.flush()                                        # = result of the second call
                    same = bool(torch.equal(s3, s) and torch.equal(i3, ids) and torch.equal(s4, s) and torch.equal(i4, ids))
                    res["pipelined_exchange_equals_complete"] = same
                    if not same:
                        raise AssertionError("pipelined exchange result differs from the complete exchange")
            if self.bm25_mode:                            # BM25 scores are produced on the device: no independent rows
                res.update({"ok": True, "note": "checker skipped for device-BM25 sparse fields"})
                return res
            n = min(n_check, qv.shape[0])
            q, spn = qv[:n], (None if sp is None else sp[:n])
            F = self.n_dense + self.n_sparse
            prev = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = False
            w = torch.softmax(q.float() @ self.layer.weight.detach().float(), dim=1) * self.retr.mask.reshape(1, F)
            torch.backends.cuda.matmul.allow_tf32 = prev
            chk = Fp32Checker(self.pc, n_docs=self.hi - self.lo, doc_id_base=self.lo)
            K2 = TOPK + 28
            cs, ci = chk.topk(q if self.pc is not None else None, w.contiguous(), TOPK, sparse=spn, slack=K2 - TOPK)
            got_i = ids[:n]
            mine = (got_i >= self.lo) & (got_i < self.hi)
            resc = chk.rescore(q if self.pc is not None else None, w.contiguous(), got_i, sparse=spn) * mine
            if ctx.world > 1:
                if cs.shape[1] < K2:                       # tiny shard: pad
                    pad = K2 - cs.shape[1]
                    cs = torch.nn.functional.pad(cs, (0, pad), value=float("-inf"))
                    ci = torch.nn.functional.pad(ci, (0, pad), value=-1)
                all_s = [torch.empty_like(cs) for _ in range(ctx.world)]
                all_i = [torch.empty_like(ci) for _ in range(ctx.world)]
                ctx.dist.all_gather(all_s, cs.contiguous())
                ctx.dist.all_gather(all_i, ci.contiguous())
                cs, ci = Fp32Checker._reduce(torch.cat(all_s, dim=1), torch.cat(all_i, dim=1), K2)
                ctx.dist.all_reduce(resc)
            if ctx.rank == 0:
                assert_topk_parity_at_scale(s[:n], got_i, cs, ci, resc, TOPK, self.n_total, 0, what=self.name)
            res.update({"queries": n, "ok": True,
                        "checker": "tests/checker.py: torch fp32 over the packed corpus, TF32 off; near-tie rule"})
        except AssertionError as e:
            res.update({"ok": False, "error": str(e)[:300]})
        return res

    # ------------------------------------------------------------------ the reference-faithful mode (SURVEY 8f-1)
    def time_union_rescore(self, Q, steps, warmup):
        """trec_eval_step as the reference runs it - per-field top-100, union, rescore, mixture, top-100 - on the device:
        one streaming top-k pass per field + ONE union/rescore kernel for the batch (mfar_union_rescore).  Also reports
        how much of the exhaustive top-100 the candidate-union pipeline recovers (it is an approximation of it)."""
        pool = self.make_batches(Q, 2)
        run = lambda b: self.retr.union_rescore_batch(b[0], b[1], b[2], TOPK)      # noqa: E731
        for i in range(warmup):
            run(pool[i % len(pool)])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            vals, rows, usize = run(pool[i % len(pool)])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        launches = self.retr.last_launches
        b = pool[(steps - 1) % len(pool)]
        _, ids = self.retr.search(b[0], b[1], b[2])
        overlap = [(len(set(rows[i].tolist()) & set((ids[i] - self.lo).tolist())) / TOPK) for i in range(min(Q, 16))]
        return {"mode": "union_rescore (reference-faithful trec_eval_step on the device)", "batch": Q,
                "value": Q * steps / (ms * 1e-3), "ms_per_step": ms / steps, "gpu_launches_per_step": launches,
                "mean_union_size": float(usize.float().mean().item()),
                "overlap_with_exhaustive_top100": sum(overlap) / len(overlap)}

    def release(self):
        self.graphs.clear()
        self.retr = self.sharded = self.piped = self.pc = self.pc_held = self.bm25_fields = None
        gc.collect()
        torch.cuda.empty_cache()


def run_workload(ctx: Ctx, name, batches, steps, warmup, headline=False):
    """All legs of one workload.  `batches[0]` is the main batch; returns a dict (rank 0 fills the line from it)."""
    a = ctx.args
    wl = Workload(ctx, name, a.docs if headline else 0)
    graph = bool(a.graph) or ctx.world > 1             # the sharded step is launch-sensitive: always replay it as a graph
    if wl.margin:
        t0 = time.perf_counter()
        wl.tune_boundaries(batches[0])
        wl.setup_s += time.perf_counter() - t0
    out = {"workload": name, "n_docs": wl.n_total, "n_dense": wl.n_dense, "n_sparse": wl.n_sparse,
           "shard_docs": wl.hi - wl.lo, "cuda_graph": graph, "setup_s": wl.setup_s, "batches": []}
    if wl.tuning:
        out["boundary_tuning"] = {"margin_docs": wl.margin, "rounds": wl.tuning,
                                  "note": "untimed start-up: per-rank scoring-kernel ms of the real sharded step, "
                                          "boundaries moved towards equal time within the resident margins"}
    for bi, Q in enumerate(batches):
        main = headline and bi == 0
        st, wu = (steps, warmup) if main else (max(5, steps // 2), 3)
        pool = wl.make_batches(Q, 4 if main else 2)
        if not main:
            # Side legs with sub-millisecond steps: ten steps after three warm-ups are ~10 ms in whatever clock / power
            # state the previous leg left behind (seen: the same PRIME-shaped kernel at 0.88 ms right after the 1 kW
            # headline leg, 0.63 ms on its own).  Size them by TIME instead: >= 40 ms of warm-up, >= 100 ms timed.
            est = wl.time_device(pool, 3, 2, graph, profile=False)[0] / 3
            st = max(st, min(300, int(math.ceil(100.0 / max(est, 1e-3)))))
            wu = max(wu, min(100, int(math.ceil(40.0 / max(est, 1e-3)))))
        keep = main and a.dump_outputs is not None
        ms, launches, km, clocks = wl.time_device(pool, st, wu, graph, profile=True, sample_clocks=main, keep_last=keep)
        if keep:
            out["last_outputs"] = wl.last_outputs
        k_ms = statistics.mean(km) if km else None
        rec = {"batch": Q, "value": Q * st / (ms * 1e-3), "ms_per_step": ms / st, "steps": st,
               "roofline": wl.roofline(Q, k_ms, len(km), ms, st), "gpu_launches": launches}
        if ctx.world > 1:
            rec["per_rank"] = {"ms_per_step": wl.last_per_rank_ms_per_step, "kernel_ms": wl.last_per_rank_kernel_ms,
                               "note": "ms_per_step: each rank's own CUDA-event time of the timed loop / steps (the line's "
                                       "ms_per_step is their maximum); kernel_ms: each rank's mean scoring-kernel time"}
        if main:
            rec["clocks"] = clocks
            ms_e, h2d, d2h = wl.time_e2e(pool, st, warmup, graph)
            rec["e2e"] = {"value": Q * st / (ms_e * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": h2d,
                          "d2h_bytes_per_step": d2h, "ms_per_step": ms_e / st,
                          "path": "mfar_search_host (C ABI, pinned host buffers)" if ctx.world == 1 else
                                  "pinned host -> device copies + sharded step (graph replay) + D2H of the merged top-k"
                                  + (" of the previous step (pipelined exchange)" if ctx.pipelined else "")}
        if Q == max(batches):                          # check the largest batch (up to 4 of its queries)
            out["parity_check"] = wl.parity_check(pool[0])
        out["batches"].append(rec)
        del pool
        gc.collect()
        torch.cuda.empty_cache()
    if ctx.world == 1 and not wl.bm25_mode and name in ("prime_full", "amazon_full", "mag_full"):
        try:
            out["union_rescore"] = wl.time_union_rescore(64, max(5, steps // 2), 3)
        except Exception as e:  # noqa: BLE001
            out["union_rescore"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    wl.release()
    return out


def dump_outputs(out_dir, scores, ids):
    """`--dump-outputs`: DIR/topk_scores.npy (float32 [Q, 100]) and DIR/topk_ids.npy (float64 [Q, 100]; doc ids are
    exact below 2**53).  Within DUMP_BYTES in all: a larger batch is cut to its first queries, a fixed sample since
    the batch is one seeded random draw."""
    import numpy as np
    n = min(scores.shape[0], (DUMP_BYTES - 4096) // (scores.shape[1] * (4 + 8)))     # 4096: room for the .npy headers
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "topk_scores.npy"), scores[:n].numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "topk_ids.npy"), ids[:n].numpy().astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="scale_10m_all")
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--docs", type=int, default=0, help="override the headline workload's doc count (debug)")
    ap.add_argument("--kernel", default="auto", choices=["auto", "simt", "tcgen05", "tcgen05_qs"])
    ap.add_argument("--extra-batches", default="1,64", help="also measured on the headline corpus (device-resident)")
    ap.add_argument("--others", default="default",
                    help="'default' = the BASELINE.json configs that ride along (C2, C3, C4, C5 single_), 'none', or a "
                         "list like mag_full:1:512,amazon_full:64")
    ap.add_argument("--sparse-mode", default="precomputed", choices=["precomputed", "bm25"],
                    help="sparse fields as precomputed [Q,Fs,N] f16 score tensors (north_star (2)) or scored on the "
                         "device from query tokens against HBM-resident BM25 postings (SURVEY 8f-3)")
    ap.add_argument("--graph", action="store_true",
                    help="N=1: replay the device-resident step as one CUDA graph (always on for N>1)")
    ap.add_argument("--balance", default="off", choices=["auto", "static", "off"],
                    help="N>1: off = equal doc ranges (default: under the node's power cap the per-GPU speed FLUCTUATES "
                         "by several per cent from one 50 ms window to the next rather than differing persistently, and "
                         "both tuners below chase that noise - measured 79.5k q/s tuned vs 81.0k equal at N=8, "
                         "profiles/r2_bench_n8_tuned_vs_equal.md); auto = every rank holds a 6 %% margin of its "
                         "neighbours' docs and the boundaries are tuned on the real step at start-up; static = one "
                         "calibration run sizes the ranges")
    ap.add_argument("--exchange-mode", default="complete", choices=["pipelined", "complete"],
                    help="N>1 timed loops: a step merges the previous step's keys (pipelined, no waiting for the slowest "
                         "rank of the step) or its own (complete)")
    ap.add_argument("--cpu-budget-s", type=float, default=20.0, help="0 skips the cpu_baseline leg of our arm")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the headline's last timed step returned (top-k scores "
                         "and doc ids) as DIR/<name>.npy; the inputs depend only on the arguments, so two builds run "
                         "with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's outputs (--impl ours)")
    args.warmup = max(args.warmup, 3)

    from mfar_b200 import synth
    n_total, n_dense, n_sparse = synth.SHAPES[args.workload]
    if args.docs:
        n_total = args.docs
    Q = args.batch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    config = {"workload": f"{args.workload}: {n_total} docs x {n_dense} dense + {n_sparse} sparse fields x {DIM}-d bf16, "
                          f"exhaustive hybrid top-{TOPK}, query-conditioned mixture",
              "n_docs": n_total, "n_dense": n_dense, "n_sparse": n_sparse, "dim": DIM, "batch": Q, "top_k": TOPK,
              "sharding": f"doc-range x{world}"}
    shard_mb = (n_total // world) * max(n_dense, 1) * DIM * 2 / 1e6
    config["cache"] = (f"corpus shard {shard_mb:.0f} MB >> 126 MB L2 (inputs larger than L2)" if shard_mb > 2 * 126 else
                       f"corpus shard {shard_mb:.0f} MB is NOT larger than the 126 MB L2 and is not flushed between steps: "
                       "small-workload numbers are L2-assisted")
    if n_sparse:
        config["sparse_input"] = ("device BM25: query tokens -> postings scatter-add (mfar_score_topk_bm25)"
                                  if args.sparse_mode == "bm25" else
                                  "precomputed [Q,Fs,N] f16 score tensor, gathered inside the scoring epilogue")

    # ------------------------------------------------------------------ reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return
        cb = cpu_reference_leg(n_total, n_dense, n_sparse, Q, args.seed, args.steps, args.warmup)
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "queries/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step_sample"],
                "ms_per_step_is": "one timed step = the bounded sample described in cpu_baseline.sample",
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm
    # Native libraries (NCCL's version banner, ...) write to fd 1; the contract is ONE JSON line on stdout, so fd 1
    # points at stderr until that line is printed.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA sm_100 device (there is no CPU fallback for the product path)")
    ctx = Ctx(args)
    if world > 1 and args.balance == "static" and n_dense:
        ctx.calibrate(n_dense, Q, n_total // world)
    if world > 1 and args.balance == "auto":
        ctx.balance_note = "boundaries tuned at start-up on the measured per-rank step time (boundary_tuning)"
    config["sharding"] = f"doc-range x{world}, {ctx.balance_note}"

    extra = [int(x) for x in args.extra_batches.split(",") if x and int(x) != Q]
    head = run_workload(ctx, args.workload, [Q] + extra, args.steps, args.warmup, headline=True)
    if rank == 0 and args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, *head["last_outputs"])
    others = []
    if args.others != "none":
        spec = OTHER_WORKLOADS if args.others == "default" else tuple(
            (s.split(":")[0], tuple(int(x) for x in s.split(":")[1:])) for s in args.others.split(",") if s)
        for name, batches in spec:
            if name == args.workload:
                continue
            try:
                others.append(run_workload(ctx, name, list(batches), args.steps, args.warmup))
            except Exception as e:  # noqa: BLE001  (a side workload must not take the headline down)
                others.append({"workload": name, "error": f"{type(e).__name__}: {e}"[:300]})

    cpu_base = None
    if rank == 0 and world == 1 and args.cpu_budget_s > 0:
        cpu_base = cpu_reference_leg(n_total, n_dense, n_sparse, Q, args.seed, 3, 1)

    if rank == 0:
        main_rec = head["batches"][0]

        def compact(rec):
            r = rec.get("roofline") or {}
            return {"batch": rec["batch"], "value": rec["value"], "ms_per_step": rec["ms_per_step"],
                    "kernel": r.get("kernel"), "kernel_ms": r.get("kernel_ms"), "bound": r.get("bound"),
                    "achieved": r.get("achieved"), "unit": r.get("unit"), "frac": r.get("frac"),
                    "frac_of_burst_peak": r.get("frac_of_burst_peak"),
                    "kernel_share_of_step": r.get("kernel_share_of_step"), "gpu_launches": rec["gpu_launches"]}
        line = {
            "metric": METRIC, "value": main_rec["value"], "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main_rec["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config,
            "roofline": main_rec["roofline"], "cpu_baseline": cpu_base, "e2e": main_rec["e2e"],
            "parity_check": head["parity_check"], "gpu_launches": main_rec["gpu_launches"],
            "exchange": ctx.exchange_kind + ("; timed loops PIPELINED: each step pushes its keys and merges the previous "
                                             "step's (results trail by one step)" if ctx.pipelined else ""),
            "clocks": main_rec["clocks"],
            "per_rank": main_rec.get("per_rank"),
            "boundary_tuning": head.get("boundary_tuning"),
            "other_batches": [compact(r) for r in head["batches"][1:]],
            "other_workloads": [
                o if "error" in o else
                {"workload": o["workload"], "n_docs": o["n_docs"], "n_dense": o["n_dense"], "n_sparse": o["n_sparse"],
                 "shard_docs": o["shard_docs"], "parity_check": o["parity_check"],
                 "batches": [compact(r) for r in o["batches"]], "union_rescore": o.get("union_rescore")}
                for o in others],
            "setup_s": head["setup_s"], "kernel_impl": args.kernel, "cuda_graph": head["cuda_graph"],
        }
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
