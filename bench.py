#!/usr/bin/env python
"""bench.py — queries/sec of FLMR late-interaction MaxSim + top-k over a 1M-passage corpus.

    python bench.py --gpus 1 --steps K --warmup W            # this repository's CUDA path
    python bench.py --impl reference ...                     # the reference's CPU path (host cores)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2] / north_star): synthetic L2-normalised bf16 embeddings,
N = 1,000,000 passages x Nd = 180 tokens x d = 128, queries of Nq = 320 tokens, k = 5.  At N GPUs the
passage-token matrix is sharded by contiguous passage ranges (1M / N per GPU: STRONG scaling), each
rank scans its shard, one NCCL all-gather of per-shard top-k, merge.

One "step" = one call of the hot path on a batch of `--batch` queries.  `value` = whole-job
queries/sec with the query batch already resident in HBM; `e2e` = the same through the
reference-facing `Searcher._search_all_Q` with the query batch in pinned HOST memory and the ranking
returned as Python lists (H2D + D2H inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "queries/sec MaxSim+top-k over 1M-passage corpus (Nq=320, Nd=180, d=128)"
UNIT = "queries/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--passages", type=int, default=1_000_000)
    ap.add_argument("--nd", type=int, default=180)
    ap.add_argument("--nq", type=int, default=320)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--k", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the baseline sample")
    ap.add_argument("--no-plaid-baseline", action="store_true")
    ap.add_argument("--plaid-passages", type=int, default=50_000,
                    help="passages in the sample PLAID index of the PLAID CPU-search baseline leg")
    ap.add_argument("--plaid-ndocs", type=int, default=1024, help="ndocs of the PLAID leg (reference default 1024)")
    ap.add_argument("--no-c2", action="store_true", help="skip the C2-shaped (112k ragged passages, Nq=832, k=100) record")
    ap.add_argument("--c2-passages", type=int, default=112_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the ranking of the last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        # the reference arm sizes its passage sample from a timing probe, so its inputs vary from run to run
        ap.error("--dump-outputs needs --impl ours")
    return args


def dump_outputs(out_dir, arrays):
    """Write each array as <out_dir>/<name>.npy: scores in float32, passage ids in float64 (exact below 2^53)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(args, world):
    """The `config` object of the JSON line — built by ONE function for both arms (`--impl ours` and
    `--impl reference`), so the driver compares like with like; arm-specific detail lives in other keys."""
    return {"workload": "FLMR MaxSim top-%d: %d passages x Nd=%d, Nq=%d, d=128, batch %d queries/step"
                        % (args.k, args.passages, args.nd, args.nq, args.batch),
            "n_passages": args.passages, "nd": args.nd, "nq": args.nq, "dim": 128, "k": args.k,
            "batch": args.batch, "parallelism": "passage-shard x%d + allgather(top-k)" % world,
            "l2": "inputs larger than L2 (%.1f GB of passage tokens per GPU per pass)"
                  % (args.passages * args.nd * 256 / world / 1e9)}


def kernel_source_sha():
    """Hash of the scan kernel's sources: the committed ncu traffic figure is only reported while it matches."""
    import hashlib
    h = hashlib.sha256()
    for fn in ("flmr_scan_kernel.cuh", "flmr_device.cuh"):
        with open(os.path.join(ROOT, "retrieval-augmented-visual-question-answering_b200", "csrc", fn), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_burst": float(p["bf16_tflops"]),
                "bf16_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "source": "fallback"}


# --------------------------------------------------------------------------------------------------
# reference CPU leg (oracle/_ref when the reference's segmented_maxsim.cpp was compiled, else the
# oracle port).  TEST/BASELINE INFRASTRUCTURE: never on the product path.
# --------------------------------------------------------------------------------------------------
def make_cpu_scorer():
    """Returns (kind, fn(Q [nq,d] fp32 torch, D [T,d] fp32 torch, doclens int64 torch) -> scores [n])."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import build_ref
        mod = build_ref.load()
    except Exception:
        mod = None
    if mod is not None:
        def ref_fn(Q, D, doclens):
            # colbert_score_packed, CPU branch (third_party/ColBERT/colbert/modeling/colbert.py:304,311):
            #   scores = D_packed @ Q.T ; ColBERT.segmented_maxsim(scores, D_lengths)
            return mod.segmented_maxsim_cpp((D @ Q.T).contiguous(), doclens)
        return "reference (its segmented_maxsim.cpp compiled in place + the D_packed @ Q.T it calls)", ref_fn
    from oracle import maxsim_oracle as O

    def port_fn(Q, D, doclens):
        return torch.from_numpy(O.colbert_score_packed(Q.numpy()[None], D.numpy(), doclens.numpy()))
    return "port", port_fn


def cpu_reference_rate(args, target_seconds, steps=1, warmup=0):
    """queries/sec of the reference's exhaustive CPU MaxSim extrapolated to the full corpus from a
    bounded sample of passages (the fp32 corpus would be 92 GB).  Returns dict for `cpu_baseline`."""
    import torch
    kind, fn = make_cpu_scorer()
    # all the host cores the box has.  torch's default (physical cores) is the fastest setting for the
    # reference's MKL GEMM + pthread reduction (SMT siblings slow it down: 0.0166 q/s at 64 threads vs
    # 0.0103 at 128 on the round-1 box); torchrun exports OMP_NUM_THREADS=1, which would cripple it
    # (segmented_maxsim.cpp spawns at::get_num_threads() threads), so undo that.
    try:
        if os.environ.get("OMP_NUM_THREADS") == "1" or torch.get_num_threads() == 1:
            torch.set_num_threads(max(1, len(os.sched_getaffinity(0)) // 2))
    except Exception:
        pass
    cores = torch.get_num_threads()
    g = torch.Generator().manual_seed(0)
    n_q = 2
    Qs = torch.nn.functional.normalize(torch.randn(n_q, args.nq, 128, generator=g), dim=-1).bfloat16().float()
    Q = Qs[0]

    def make(n):
        D = torch.nn.functional.normalize(torch.randn(n * args.nd, 128, generator=g), dim=-1).bfloat16().float()
        return D, torch.full((n,), args.nd, dtype=torch.int64)

    n_probe = 2000
    D, dl = make(n_probe)
    fn(Q, D, dl)                                   # warm caches / thread pools
    t0 = time.perf_counter()
    fn(Q, D, dl)
    t_probe = time.perf_counter() - t0
    n_sample = int(min(max(n_probe, n_probe * target_seconds / max(t_probe * n_q, 1e-4)), 100_000, args.passages))
    D, dl = make(n_sample)
    for _ in range(warmup):
        fn(Q, D, dl)
    times = []
    for _ in range(max(steps, 1)):
        t0 = time.perf_counter()
        for qi in range(n_q):                       # the reference scores one query at a time (colbert.py:297)
            s = fn(Qs[qi], D, dl)
            s.topk(min(args.k, n_sample))
        times.append(time.perf_counter() - t0)
    t_step = sum(times) / len(times)
    per_query_full = (t_step / n_q) * (args.passages / n_sample)
    return {"value": 1.0 / per_query_full, "unit": UNIT, "cores": cores, "kind": kind,
            "sample_fraction": n_sample / args.passages, "sample_queries": n_q,
            "sample": "%d queries x %d of %d passages (Nq=%d, Nd=%d) exhaustive colbert_score_packed + topk, "
                      "%.2f s per step, per-query time linearly extrapolated to the full corpus" %
                      (n_q, n_sample, args.passages, args.nq, args.nd, t_step),
            "ms_per_step": t_step * 1e3}


def cpu_plaid_rate(args, device, target_seconds=10.0):
    """queries/sec of the reference's PLAID CPU search (what FLMR_executor.py:778-792 runs under DDP):
    oracle/plaid_search.py = restated glue + the reference's own compiled kernels (oracle/_ref), or the
    restatements of those kernels where they were not built (kind "port").

    A PLAID index of the full 1M x 180 corpus is a ~6.5 GB build; the leg is bounded to a clustered sample
    of `--plaid-passages` passages (index build on `device`, outside the timed region) and says so: PLAID's
    candidate lists grow with the corpus, so the figure is an UPPER bound of its rate at 1M passages.
    PLAID returns an approximate ranking; the exhaustive legs return the exact one."""
    import torch
    from oracle import plaid_search as P
    try:
        if os.environ.get("OMP_NUM_THREADS") == "1" or torch.get_num_threads() == 1:
            torch.set_num_threads(max(1, len(os.sched_getaffinity(0)) // 2))
    except Exception:
        pass
    n, nd, nq, nbits = args.plaid_passages, args.nd, args.nq, 2
    n_emb = n * nd
    K = int(2 ** math.floor(math.log2(16 * math.sqrt(n_emb))))   # collection_indexer.py:93
    dev = torch.device(device)
    g = torch.Generator(device=dev).manual_seed(1234)
    t0 = time.perf_counter()
    # clustered synthetic tokens: topic direction + per-dimension noise 0.06 (token/topic cosine ~0.83,
    # residual norms in the range real ColBERT indexes show); 256 topics, 3 per passage, so the
    # candidate list of a query grows linearly with the corpus (~1.2 % of the passages per topic).
    n_topics = 256
    topics = torch.nn.functional.normalize(torch.randn(n_topics, 128, generator=g, device=dev), dim=-1)
    ptop = torch.randint(0, n_topics, (n, 3), generator=g, device=dev)
    pick = torch.randint(0, 3, (n, nd), generator=g, device=dev)
    tok_topic = torch.gather(ptop, 1, pick).flatten()
    D = torch.empty(n_emb, 128, dtype=torch.bfloat16, device=dev)
    for a in range(0, n_emb, 1 << 20):
        b = min(n_emb, a + (1 << 20))
        D[a:b] = torch.nn.functional.normalize(
            topics[tok_topic[a:b]] + 0.06 * torch.randn(b - a, 128, generator=g, device=dev), dim=-1).bfloat16()
    doclens = torch.full((n,), nd, dtype=torch.long)
    sample = D[torch.randperm(n_emb, generator=g, device=dev)[: min(n_emb, 8 * K)]].float()
    centroids = P.train_centroids(sample.cpu(), K, iters=4, seed=0, device=dev)
    index = P.PlaidIndex.build(D, doclens, centroids, nbits, heldout=sample[: 1 << 16], device=dev)
    # queries: Nq noisy tokens of a planted passage (the first query_maxlen=32 select the cells, all Nq score)
    n_queries = 64
    targets = torch.randint(0, n, (n_queries,), generator=g, device=dev)
    rows = torch.randint(0, nd, (n_queries, nq), generator=g, device=dev) + (targets * nd).unsqueeze(1)
    Q = torch.nn.functional.normalize(D[rows.flatten()].float().view(n_queries, nq, 128)
                                      + 0.04 * torch.randn(n_queries, nq, 128, generator=g, device=dev), dim=-1)
    Q = Q.bfloat16().float().cpu()
    targets = targets.cpu().tolist()
    del D, sample
    t_build = time.perf_counter() - t0
    searcher = P.PlaidSearcher(index)
    kw = dict(ncells=2, threshold=0.45, ndocs=getattr(args, "plaid_ndocs", 1024), query_maxlen=32)      # colbert/searcher.py:100-103 (k <= 10)
    n_cand = []
    for i in range(2):                                                     # warm-up + candidate-count check
        cand, _ = searcher.retrieve(Q[i:i + 1], kw["ncells"], kw["query_maxlen"])
        n_cand.append(int(cand.numel()))
    if min(n_cand) < kw["ndocs"]:
        return {"value": None, "unit": UNIT, "kind": "unavailable",
                "sample": "only %d candidates < ndocs=%d on a %d-passage sample: filter_pids.cpp is undefined there"
                          % (min(n_cand), kw["ndocs"], n)}
    searcher.rank(Q[0:1], **kw)
    hits, done, t_total = 0, 0, 0.0
    for i in range(n_queries):
        t1 = time.perf_counter()
        pids, _ = searcher.rank(Q[i:i + 1], **kw)
        t_total += time.perf_counter() - t1
        hits += int(targets[i] in pids[: args.k])
        done += 1
        if t_total > target_seconds:
            break
    return {"value": done / t_total, "unit": UNIT, "cores": torch.get_num_threads(),
            "kind": "reference" if searcher.compiled else "port",
            "ms_per_query": 1e3 * t_total / done, "recall_at_%d" % args.k: hits / done,
            "candidates_per_query": n_cand, "index": {"passages": n, "centroids": K, "nbits": nbits,
                                                      "build_seconds": t_build, "build_device": str(dev)},
            "sample": "%d queries (Nq=%d, first 32 tokens select cells) through the restated IndexScorer.rank "
                      "(ncells=2, centroid_score_threshold=0.45, ndocs=%d) over a clustered %d-passage x Nd=%d "
                      "PLAID index, nbits=2; NOT extrapolated to 1M passages (candidate lists grow with the corpus), "
                      "approximate ranking" % (done, nq, kw["ndocs"], n, nd)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base = cpu_reference_rate(args, target_seconds=max(2.0, min(args.cpu_seconds, 20.0)),
                              steps=args.steps, warmup=min(args.warmup, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, max(1, args.gpus)),
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "sample_fraction",
                                              "sample_queries")},
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    # also report the reference's PRUNED search (what its executors actually run; approximate ranking) when a
    # GPU is there to build the sample PLAID index quickly with torch ops — the timed search itself is CPU-only
    if not args.no_plaid_baseline:
        try:
            import torch
            if torch.cuda.is_available():
                line["cpu_baseline_plaid"] = cpu_plaid_rate(args, "cuda:0")
        except Exception as e:
            line["cpu_baseline_plaid"] = {"value": None, "unit": UNIT, "kind": "error", "sample": repr(e)}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# this repository's arm
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.QUERY,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, smax, power, reasons = [], [], [], set()
        for line in self.f.read().strip().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
                power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                 parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


CHUNK = 20_000   # passages per generation chunk; chunk boundaries are GLOBAL so any rank can regenerate any passage


def gen_chunk(ci, nd, dev):
    """bf16 [CHUNK * nd, 128]: the tokens of global passages [ci * CHUNK, (ci + 1) * CHUNK), seeded by ci."""
    import torch
    g = torch.Generator(device=dev).manual_seed(1_000_003 * ci + 17)
    x = torch.randn((CHUNK * nd, 128), device=dev, generator=g)
    return torch.nn.functional.normalize(x, dim=-1).to(torch.bfloat16)


def build_shard(p0, p1, nd, dev):
    import torch
    D = torch.empty(((p1 - p0) * nd, 128), dtype=torch.bfloat16, device=dev)
    for ci in range(p0 // CHUNK, (p1 + CHUNK - 1) // CHUNK):
        a, b = max(p0, ci * CHUNK), min(p1, (ci + 1) * CHUNK)
        D[(a - p0) * nd:(b - p0) * nd] = gen_chunk(ci, nd, dev)[(a - ci * CHUNK) * nd:(b - ci * CHUNK) * nd]
    return D


def planted_queries(B, nq, nd, n_total, world, dev):
    """Query b = Nq noisy copies (token/query cosine ~0.83) of the tokens of ONE corpus passage t_b that lives in
    shard b mod world: a known positive per query, each in a different shard, so the MERGED global top-k of the
    sharded search can be asserted at every N (and Recall@k reported).  The kernel's work is data-independent."""
    import torch
    targets, rows = [], []
    for b in range(B):
        r = b % world
        s0, s1 = n_total * r // world, n_total * (r + 1) // world
        t = s0 + (7919 * (b + 1)) % (s1 - s0)
        ci = t // CHUNK
        tok = gen_chunk(ci, nd, dev)[(t - ci * CHUNK) * nd:(t - ci * CHUNK + 1) * nd].float()
        rows.append(tok[torch.arange(nq, device=dev) % nd])
        targets.append(t)
    g = torch.Generator(device=dev).manual_seed(12345)
    Q = torch.stack(rows)
    Q = torch.nn.functional.normalize(Q + 0.06 * torch.randn(Q.shape, device=dev, generator=g), dim=-1)
    return Q, targets


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import ravqa_b200 as R
    from ravqa_b200 import _cabi
    import ctypes as C

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun with that many ranks" % args.gpus)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner to STDOUT at NCCL_DEBUG=VERSION; stdout must carry exactly one
        # JSON line
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # whatever NCCL still says goes to stderr
        dist.init_process_group("nccl", device_id=dev)

    # ---- this rank's shard of the synthetic corpus, generated on-device ----
    n_total, nd, nq, B, k = args.passages, args.nd, args.nq, args.batch, args.k
    p0 = n_total * rank // world
    p1 = n_total * (rank + 1) // world
    n_local = p1 - p0
    D = build_shard(p0, p1, nd, dev)
    corpus = R.FlatCorpus(D, np.full(n_local, nd, dtype=np.int32), device=dev, pid_base=p0)
    # queries with a planted positive each (rank 0 builds them, everyone receives the same bits)
    if rank == 0:
        Q32, targets = planted_queries(B, nq, nd, n_total, world, dev)
    else:
        Q32, targets = torch.empty((B, nq, 128), device=dev), [0] * B
    if world > 1:
        dist.broadcast(Q32, src=0)
    Q_host = Q32.cpu().pin_memory()                  # fp32, pinned: what an encoder hands the Searcher
    Q_dev = Q32.to(torch.bfloat16)
    # THE product path: the reference-facing Searcher; with N ranks it keeps this rank's shard and merges the
    # per-shard top-k with one all-gather
    searcher = R.Searcher(index=corpus, shard_across_ranks=(world > 1))
    L = _cabi.lib()
    qids = list(range(B))

    def step_device():
        return searcher._search_tensors(Q_dev, k)

    def step_e2e():
        return searcher._search_all_Q(qids, Q_host, k, progress=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, warmup, profile=False, clocks=True):
        for _ in range(warmup):
            fn()
        barrier()
        if profile:
            L.flmr_scan_kernel_stats(None, None, 1)
            L.flmr_set_profiling(1)
        L.flmr_launch_count(1)
        sampler = ClockSampler(local_rank) if (rank == 0 and clocks) else None
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        dev_ms = e0.elapsed_time(e1)
        clk = sampler.stop() if sampler else None
        launches = int(L.flmr_launch_count(0))
        scan_ms, scan_n = C.c_double(0), C.c_int64(0)
        if profile:
            L.flmr_scan_kernel_stats(C.byref(scan_ms), C.byref(scan_n), 1)
            L.flmr_set_profiling(0)
        t = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return {"dev_ms": t[0].item(), "wall_ms": t[1].item(), "clocks": clk, "launches": launches,
                "scan_ms": scan_ms.value, "scan_n": scan_n.value, "out": out}

    # device-resident timing (value) with per-launch scan-kernel events for the roofline
    r_dev = timed(step_device, args.steps, args.warmup, profile=True)
    ms_per_step = r_dev["dev_ms"] / args.steps
    value = B * 1e3 / ms_per_step
    # end-to-end through the reference-facing API with host buffers (wall clock spans H2D/D2H/lists)
    r_e2e = timed(step_e2e, args.steps, min(args.warmup, 2))
    e2e_ms = max(r_e2e["dev_ms"], r_e2e["wall_ms"]) / args.steps
    e2e_value = B * 1e3 / e2e_ms

    # ---- parity inside the bench ----
    # (1) the MERGED global ranking: every query's planted positive (each in a different shard) must come out
    #     first, on every rank; Recall@k = share of queries whose positive is in the returned top-k
    m_scores, m_pids = r_dev["out"]
    pid_rows = m_pids.cpu().tolist()
    if world > 1:
        tg = torch.tensor(targets, dtype=torch.int64, device=dev)
        dist.broadcast(tg, src=0)
        targets = tg.tolist()
    recall_1 = sum(int(row[0] == t) for row, t in zip(pid_rows, targets)) / B
    recall_k = sum(int(t in row) for row, t in zip(pid_rows, targets)) / B
    e2e_ranking = r_e2e["out"].todict()
    e2e_rows = [[p for p, _, _ in e2e_ranking[q]] for q in qids]
    e2e_same = e2e_rows == pid_rows
    if args.dump_outputs and rank == 0:
        # the merged global top-k of the last timed step of each timed path (identical on every rank)
        dump_outputs(args.dump_outputs, {
            "topk_scores": m_scores.float().cpu().numpy(),
            "topk_pids": np.asarray(pid_rows, dtype=np.float64),
            "e2e_scores": np.asarray([[s for _, _, s in e2e_ranking[q]] for q in qids], dtype=np.float32),
            "e2e_pids": np.asarray(e2e_rows, dtype=np.float64)})
    # (2) the fused result equals top-k of the all-scores path on this shard
    s_all = R.maxsim_scores(corpus, Q_dev[:1])
    ts, tp = R.maxsim_topk(corpus, Q_dev[:1], k)
    rs, rp = torch.sort(s_all, dim=1, descending=True, stable=True)
    self_check = bool(torch.equal(tp, rp[:, :k] + p0))
    del s_all, rs, rp

    def scan_only(Qx, kk, reps):
        """Average CUDA-event time of the scan launches of `reps` searches (warm)."""
        for _ in range(2):
            R.maxsim_topk(corpus, Qx, kk)
        torch.cuda.synchronize(dev)
        L.flmr_scan_kernel_stats(None, None, 1)
        L.flmr_set_profiling(1)
        for _ in range(reps):
            R.maxsim_topk(corpus, Qx, kk)
        torch.cuda.synchronize(dev)
        tot, cnt = C.c_double(0), C.c_int64(0)
        L.flmr_scan_kernel_stats(C.byref(tot), C.byref(cnt), 1)
        L.flmr_set_profiling(0)
        return (tot.value / cnt.value) if cnt.value else None

    peaks = load_peaks()
    n_tok = float(corpus.info.n_tokens)
    hbm_regime = b1 = None
    if world == 1:
        # the same kernel in its HBM-bound regime (one query of 32 tokens per corpus pass, the C1 query shape)
        ms = scan_only(Q_dev[:1, :32].contiguous(), k, 5)
        if ms:
            gbs = n_tok * 256.0 / (ms * 1e-3) / 1e9
            hbm_regime = {"workload": "1 query x Nq=32 per corpus pass (HBM-bound regime of the same kernel)",
                          "launch_ms": ms, "achieved": gbs, "unit": "GB/s", "queries_per_s": 1e3 / ms,
                          "peak": peaks["hbm_gbs"], "frac": gbs / peaks["hbm_gbs"], "frac_of_8TBs": gbs / 8000.0}
        # the north star's own shape: ONE query of Nq=320 per corpus pass (single-query latency path)
        ms = scan_only(Q_dev[:1].contiguous(), k, 5)
        if ms:
            gbs = n_tok * 256.0 / (ms * 1e-3) / 1e9
            tf = 2.0 * nq * 128 * n_tok / (ms * 1e-3) / 1e12
            b1 = {"workload": "1 query x Nq=%d per corpus pass (batch 1: the shape the north star's HBM fraction "
                              "is defined on)" % nq,
                  "launch_ms": ms, "queries_per_s": 1e3 / ms,
                  "hbm": {"achieved": gbs, "unit": "GB/s", "frac_of_measured_copy": gbs / peaks["hbm_gbs"],
                          "hbm_frac_of_8TBs": gbs / 8000.0},
                  "tensor": {"achieved": tf, "unit": "TFLOP/s (algorithmic: %d query rows)" % nq,
                             "frac_of_burst": tf / peaks["bf16_burst"], "frac_of_sustained": tf / peaks["bf16_sustained"]},
                  "query_rows_resident": ((nq + 31) // 32) * 32, "mma_rows_issued": ((nq + 127) // 128) * 128}

    # library GPU baseline (SURVEY.md §8d): the torch/cuBLAS composition the reference's GPU branch runs —
    # colbert_score (colbert.py:268-286): D_padded @ Q^T materialised as [n, Nd, Nq], padding fill, max over
    # passage tokens, sum over query tokens — restated in bf16 over the same resident corpus, one query,
    # chunks of 20k passages (2.3 GB of scores each), then torch.topk.  Uniform doclens: the mask is all-valid
    # but the reference's fill pass is still executed.
    lib_gpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            Dv = D.view(n_local, nd, 128)
            q1 = Q_dev[0]
            pad = torch.zeros((20_000, nd), dtype=torch.bool, device=dev)

            def lib_query():
                outs = []
                for c0 in range(0, n_local, 20_000):
                    sc = Dv[c0:c0 + 20_000] @ q1.T                       # colbert.py:284
                    sc[pad[: sc.size(0)]] = -9999                        # colbert.py:239-240
                    outs.append(sc.max(1).values.sum(-1).float())        # colbert.py:241, 263
                return torch.cat(outs).topk(k)
            lib_query()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                lib_top = lib_query()
            e1.record()
            torch.cuda.synchronize(dev)
            lib_ms = e0.elapsed_time(e1) / 3
            ours_top = R.maxsim_topk(corpus, Q_dev[:1], k)[1][0] - p0
            lib_gpu = {"value": 1e3 / lib_ms, "unit": UNIT, "ms_per_query": lib_ms,
                       "kind": "torch/cuBLAS restatement of colbert_score's GPU branch (bf16, scores materialised)",
                       "top_k_overlap_with_fused_path": len(set(lib_top.indices.tolist()) & set(ours_top.tolist())) / k,
                       "sample": "1 query x all %d passages, 20k-passage chunks, 3 repetitions" % n_local}
            del Dv, pad
        except Exception as e:
            lib_gpu = {"value": None, "unit": UNIT, "kind": "error", "sample": repr(e)}

    # ---- C4-shaped record (BASELINE.json configs[3]: contrastive step, in-batch negatives, bsz 64 on 8 GPUs = 8
    # queries x 16 documents per rank, Nq = 832, Nd = 512): the MaxSim loss step (forward + backward) of one rank,
    # and with N > 1 the same with cross-rank negatives (all-gather of the documents, [8, N*16] matrix per rank,
    # all-reduce of dD; CB/modeling/colbert.py:64-113, 115-163).  Max over ranks of CUDA-event time.
    c4 = None
    try:
        c4 = c4_record(dev, world, rank)
    except Exception as e:
        c4 = {"kind": "error", "sample": repr(e)}

    # ---- C2-shaped record (BASELINE.json configs[1]: PreFLMR ViT-B on OK-VQA's 112k-passage corpus): ragged
    # passages, the full 832-row FLMR query (512 text + 320 vision rows, row-sliced over passes), k = max(Ks) = 100
    c2 = None
    if world == 1 and not args.no_c2:
        try:
            searcher = None
            corpus.close()
            del D
            torch.cuda.empty_cache()
            c2 = c2_record(args, dev, peaks)
        except Exception as e:
            c2 = {"value": None, "unit": UNIT, "kind": "error", "sample": repr(e)}

    if rank == 0:
        info_tokens = n_tok
        # dominant kernel = flmr_scan_kernel: one launch scans this rank's shard for the queries resident
        # in that pass.  Algorithmic work per launch (DESIGN.md "Roofline"):
        # queries resident per scan launch, from the launches actually timed (2 per normal pass at Nq = 320; 4 per
        # CTA-pair pass, where two CTAs stream one token range with two queries each)
        q_per_launch = B * args.steps / max(r_dev["scan_n"], 1)
        flops_launch = 2.0 * q_per_launch * nq * 128 * info_tokens
        bytes_launch = info_tokens * 256.0
        scan_avg_ms = r_dev["scan_ms"] / max(r_dev["scan_n"], 1)
        ach_tf = flops_launch / (scan_avg_ms * 1e-3) / 1e12 if scan_avg_ms > 0 else 0.0
        ach_gbs = bytes_launch / (scan_avg_ms * 1e-3) / 1e9 if scan_avg_ms > 0 else 0.0
        # DRAM traffic of one launch from the committed `ncu --set full` capture at this exact size; reported
        # only while the kernel sources still hash to what was captured (else null: stale)
        traffic = traffic_src = None
        sha = kernel_source_sha()
        for tname in ("r02_traffic.json", "r01_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", tname)
            if os.path.exists(tpath) and world == 1 and (n_total, nd, nq) == (1_000_000, 180, 320):
                with open(tpath) as f:
                    tj = json.load(f)
                if tj.get("kernel_source_sha") == sha and abs(tj.get("queries_per_launch", 2) - q_per_launch) < 1e-6:
                    traffic = tj.get("traffic_bytes_per_launch")
                    traffic_src = "profiles/%s (ncu --set full: dram__bytes_read.sum + dram__bytes_write.sum per launch; kernel sources %s)" % (tname, sha)
                    break
        roofline = {
            "bound": "tensor", "achieved": ach_tf, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
            "frac": ach_tf / peaks["bf16_sustained"], "traffic": traffic,
            "traffic_source": traffic_src, "kernel_source_sha": sha,
            "peak_source": peaks["source"] + " (sustained cuBLAS bf16: kernel timed inside a long step)",
            "kernel": "flmr_scan_kernel", "launch_ms": scan_avg_ms, "launches_timed": r_dev["scan_n"],
            "scan_share_of_step": r_dev["scan_ms"] / r_dev["dev_ms"] if r_dev["dev_ms"] > 0 else None,
            "hbm": {"achieved": ach_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": ach_gbs / peaks["hbm_gbs"], "frac_of_8TBs": ach_gbs / 8000.0,
                    "algorithmic_bytes_per_launch": bytes_launch},
            "algorithmic_flops_per_launch": flops_launch, "queries_per_launch": q_per_launch,
        }
        if hbm_regime:
            roofline["hbm_bound_regime"] = hbm_regime
        if b1:
            roofline["b1"] = b1
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args, world),
            "clocks": r_dev["clocks"],
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": B * nq * 128 * 4, "d2h_bytes_per_step": B * k * 12,
                    "api": "Searcher._search_all_Q(queries, Q_host_fp32_pinned, k) -> Ranking"},
            "gpu_launches": r_dev["launches"],
            "roofline": roofline,
            "recall_at_%d" % k: recall_k, "recall_at_1": recall_1,
            "parity": {"merged_top1_is_the_planted_positive": recall_1 == 1.0,
                       "positives": "one per query, query b's in shard b mod %d" % world,
                       "e2e_ranking_equals_device_ranking": e2e_same,
                       "fused_topk_equals_sorted_scores_on_local_shard": self_check},
            "self_check_fused_topk_equals_sorted_scores": self_check,
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                base = cpu_reference_rate(args, args.cpu_seconds)
                line["cpu_baseline"] = {kk: base[kk] for kk in ("value", "unit", "cores", "kind", "sample",
                                                                "sample_fraction", "sample_queries")}
            except Exception as e:  # the baseline must never take the bench line down
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": None, "kind": "error", "sample": repr(e)}
        if lib_gpu:
            line["library_gpu_baseline"] = lib_gpu
        if c2:
            line["c2"] = c2
        if c4:
            line["c4_loss_step"] = c4
        if world == 1 and not args.no_cpu_baseline and not args.no_plaid_baseline:
            try:
                line["cpu_baseline_plaid"] = cpu_plaid_rate(args, "cuda:%d" % local_rank)
            except Exception as e:
                line["cpu_baseline_plaid"] = {"value": None, "unit": UNIT, "kind": "error", "sample": repr(e)}
        print(json.dumps(line), flush=True)
    ok = (recall_1 == 1.0) and self_check and e2e_same
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not ok:
        raise SystemExit("bench parity check failed: recall@1=%.3f self_check=%s e2e_same=%s"
                         % (recall_1, self_check, e2e_same))


def c4_record(dev, world, rank):
    import torch
    import torch.distributed as dist
    import ravqa_b200 as R
    B, nway, nq, nd = 8, 2, 832, 512
    g = torch.Generator().manual_seed(1000 + rank)
    Q = torch.nn.functional.normalize(torch.randn(B, nq, 128, generator=g), dim=-1).to(dev).requires_grad_(True)
    D = torch.nn.functional.normalize(torch.randn(B * nway, nd, 128, generator=g), dim=-1).to(dev).requires_grad_(True)
    lens = torch.randint(nd // 2, nd + 1, (B * nway,), generator=g)
    mask = (torch.arange(nd)[None, :] < lens[:, None]).unsqueeze(-1).to(dev)

    def timed(cross, reps=20, loss_fn=None):
        def step():
            Q.grad = D.grad = None
            if loss_fn is not None:
                loss_fn(Q, D, mask).backward()
            else:
                R.in_batch_negatives_loss(Q, D, mask, nway, cross_rank_negatives=cross).backward()
        for _ in range(3):
            step()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            step()
        b.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t = torch.tensor([a.elapsed_time(b) / reps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()
    rec = {"workload": "MaxSim in-batch-negatives loss, forward + backward: %d ranks x (8 queries x 16 documents), "
                       "Nq=832, Nd=512 ragged, d=128 (bsz %d)" % (world, 8 * world),
           "local_negatives_ms": timed(False), "unit": "ms per step, max over ranks"}
    try:   # the same step with forward and backward replayed as CUDA graphs (fixed batch shape)
        rec["local_negatives_cuda_graphs_ms"] = timed(False, loss_fn=R.graphed_in_batch_negatives_loss(Q, D, mask, nway))
    except Exception as e:   # a record, not a gate: the eager figure above stands on its own
        rec["local_negatives_cuda_graphs_ms"] = None
        rec["cuda_graphs_error"] = repr(e)[:200]
    if world > 1:
        rec["cross_rank_negatives_ms"] = timed(True)
        rec["cross_rank_matrix"] = "[8, %d] per rank" % (B * nway * world)
    return rec


def c2_record(args, dev, peaks):
    """One GPU, C2 shape: `--c2-passages` ragged passages (90..180 tokens, the OK-VQA GoogleSearch corpus at
    max_decoder_source_length-ish lengths), 16 queries of Nq = 832 rows, k = 100 (max(Ks),
    FLMR_base_preload_vision_features.jsonnet:141).  Own roofline: FLOPs = 2 * B * 832 * 128 * tokens per step
    over the summed CUDA-event time of the step's scan launches."""
    import ctypes as C
    import numpy as np
    import torch
    import ravqa_b200 as R
    from ravqa_b200 import _cabi
    L = _cabi.lib()
    n, nq, k, B = args.c2_passages, 832, 100, 16
    g = torch.Generator().manual_seed(2)
    doclens = torch.randint(90, 181, (n,), generator=g)
    n_tok = int(doclens.sum())
    D = torch.empty((n_tok, 128), dtype=torch.bfloat16, device=dev)
    gd = torch.Generator(device=dev).manual_seed(3)
    for a in range(0, n_tok, 1 << 22):
        b = min(n_tok, a + (1 << 22))
        D[a:b] = torch.nn.functional.normalize(torch.randn((b - a, 128), device=dev, generator=gd), dim=-1).bfloat16()
    off = torch.cat([torch.zeros(1, dtype=torch.long), doclens.cumsum(0)])
    targets = [(104_729 * (b + 1)) % n for b in range(B)]
    rows = []
    for t in targets:                               # planted positive per query (as in the headline workload)
        tok = D[off[t]:off[t + 1]].float()
        rows.append(tok[torch.arange(nq, device=dev) % tok.size(0)])
    Q = torch.stack(rows)
    Q = torch.nn.functional.normalize(Q + 0.06 * torch.randn(Q.shape, device=dev, generator=gd), dim=-1).bfloat16()
    corpus = R.FlatCorpus(D, doclens.numpy().astype(np.int32), device=dev)
    del D
    searcher = R.Searcher(index=corpus)
    steps, warmup = max(3, min(args.steps, 10)), 3
    for _ in range(warmup):
        searcher._search_tensors(Q, k)
    torch.cuda.synchronize(dev)
    L.flmr_scan_kernel_stats(None, None, 1)
    L.flmr_set_profiling(1)
    L.flmr_launch_count(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        s, p = searcher._search_tensors(Q, k)
    e1.record()
    torch.cuda.synchronize(dev)
    launches = int(L.flmr_launch_count(0))
    tot, cnt = C.c_double(0), C.c_int64(0)
    L.flmr_scan_kernel_stats(C.byref(tot), C.byref(cnt), 1)
    L.flmr_set_profiling(0)
    ms_step = e0.elapsed_time(e1) / steps
    scan_ms_step = tot.value / steps
    flops_step = 2.0 * B * nq * 128 * n_tok
    tf = flops_step / (scan_ms_step * 1e-3) / 1e12
    rows_out = p.cpu().tolist()
    rec = {"workload": "C2 shape: %d ragged passages (90..180 tokens, %d tokens), %d queries x Nq=%d, k=%d"
                       % (n, n_tok, B, nq, k),
           "value": B * 1e3 / ms_step, "unit": UNIT, "ms_per_step": ms_step, "steps": steps, "warmup": warmup,
           "scan_launches_per_step": cnt.value // steps, "gpu_launches_per_step": launches // steps,
           "recall_at_1": sum(int(r[0] == t) for r, t in zip(rows_out, targets)) / B,
           "recall_at_100": sum(int(t in r) for r, t in zip(rows_out, targets)) / B,
           "roofline": {"bound": "tensor", "achieved": tf, "unit": "TFLOP/s", "peak": peaks["bf16_burst"],
                        "frac": tf / peaks["bf16_burst"],
                        "peak_source": peaks["source"] + " (burst cuBLAS bf16: a 50 ms step, not power-limited)",
                        "scan_ms_per_step": scan_ms_step, "scan_share_of_step": scan_ms_step / ms_step,
                        "algorithmic_flops_per_step": flops_step,
                        "hbm_gbs": (cnt.value // steps) * n_tok * 256.0 / (scan_ms_step * 1e-3) / 1e9}}
    # ---- C5-shaped record on the same corpus: the retrieval block of the RAG loop (rag_model_blip.py:388-443) for a
    # batch of 8 questions — exhaustive search of max(5, n_docs) passages, gather of their embeddings out of HBM,
    # differentiable re-score (block-diagonal launch), backward to the query embeddings
    try:
        Qr = Q[:8].float().requires_grad_(True)

        def rag_step():
            Qr.grad = None
            out = searcher.retrieve_and_rescore(Qr, 5)
            out["doc_scores"].sum().backward()
            return out
        for _ in range(3):
            out = rag_step()
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(steps):
            out = rag_step()
        e1.record()
        torch.cuda.synchronize(dev)
        ms_rag = e0.elapsed_time(e1) / steps
        ids = out["retrieved_doc_ids"]
        rec["c5_rag_retrieval_block"] = {
            "workload": "8 questions x Nq=832: search top-5 over the %d passages, gather, differentiable re-score, "
                        "backward to the queries (RagModelForBlip.main_retrieve's retrieval block)" % n,
            "ms_per_step": ms_rag, "questions_per_s": 8e3 / ms_rag,
            "top1_is_planted_positive": sum(int(ids[b][0] == targets[b]) for b in range(8)) / 8,
            "query_grad_finite": bool(torch.isfinite(Qr.grad).all())}
    except Exception as e:
        rec["c5_rag_retrieval_block"] = {"kind": "error", "sample": repr(e)}
    corpus.close()
    return rec


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
