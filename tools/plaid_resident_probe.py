"""Compressed (PLAID residency) vs decoded (bf16) scans of the same seeded, device-generated PLAID-format corpus.

  python tools/plaid_resident_probe.py [--passages 1000000] [--capacity-passages 11000000] [--out FILE]

Part 1, per nbits in {2, 8}: 1M passages x 180 tokens, K = 65 536 centroids; both residencies built from the same
arrays; shapes (Nq, B) = (320, 16), (320, 1), (32, 16); compressed and decoded timed in alternating blocks within
this one process (CUDA events per scan launch via flmr_scan_kernel_stats, per call around the calls); every block
asserts identical top-k scores and ids.  Reports ms per scan launch, queries/s, algorithmic bytes per corpus pass
(the decoded path streams 256 B per row; the compressed one 8 + 16 nbits B per row from HBM plus a 512 B centroid
row per token, mostly from L2), resident HBM bytes and passages that fit per GPU.

Part 2 (capacity): 11M x 180 tokens at nbits = 2 (1.98e9 stored rows, just under the 2^31-row limit of one corpus
handle; 507 GB decoded, far more than one device holds) loaded chunk by chunk through flmr_corpus_plaid_builder_*
(each 1M-passage slice generated from its own seed, appended, freed: peak device memory = resident arrays + one
slice) and searched compressed; its top-k must equal the merge of decoded searches over the same slices, built one
at a time.  Peak device memory during the load is read from cudaMemGetInfo.

Passages per GPU = min(what fits the card's memory after 4 GiB of headroom, what fits the 2^31-row handle limit).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import ravqa_b200 as R  # noqa: E402
from ravqa_b200 import _cabi  # noqa: E402
from ravqa_b200.plaid import MAX_SHARD_ROWS, _append, _builder_from, decode_chunk  # noqa: E402

ND, K_CENT, TOPK = 180, 65536, 10


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        out = "nvidia-smi unavailable: %s" % e
    return {"query": q, "value": out, "torch_name": torch.cuda.get_device_name(0)}


def synth(n_passages, nbits, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    centroids = torch.nn.functional.normalize(torch.randn(K_CENT, 128, device=dev, generator=g), dim=-1).half().float()
    weights = (torch.sort(torch.randn(1 << nbits, device=dev, generator=g)).values * 0.05).contiguous()
    codes, residuals = synth_rows(n_passages * ND, nbits, seed + 1, dev)
    return codes, residuals, centroids, weights, np.full(n_passages, ND, dtype=np.int32)


def synth_rows(n_tok, nbits, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    codes = torch.randint(0, K_CENT, (n_tok,), device=dev, generator=g, dtype=torch.int32)
    residuals = torch.empty((n_tok, 16 * nbits), dtype=torch.uint8, device=dev)
    step = 1 << 24
    for r0 in range(0, n_tok, step):
        r1 = min(n_tok, r0 + step)
        residuals[r0:r1] = torch.randint(0, 256, (r1 - r0, 16 * nbits), device=dev, generator=g,
                                         dtype=torch.int32).to(torch.uint8)
    return codes, residuals


def passages_per_gpu(bytes_per_passage, rows_per_passage, total):
    by_memory = int((total - (4 << 30)) / bytes_per_passage)
    by_rows = int(MAX_SHARD_ROWS // rows_per_passage)
    return {"by_memory": by_memory, "by_row_limit": by_rows, "passages": min(by_memory, by_rows)}


def decoded_corpus(codes, residuals, centroids, weights, nbits, doclens, dev, pid_base=0):
    tokens = torch.empty((codes.numel(), 128), dtype=torch.bfloat16, device=dev)
    decode_chunk(codes, residuals, centroids, weights, nbits, tokens)
    return R.FlatCorpus(tokens, doclens, device=dev, pid_base=pid_base)     # aligned doclens: adopted


def compressed_corpus(codes, residuals, centroids, weights, nbits, doclens, dev, pid_base=0):
    return R.FlatCorpus.from_plaid_arrays(codes, residuals, centroids, weights, nbits, doclens, dev, pid_base)


def queries(B, nq, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.nn.functional.normalize(torch.randn(B, nq, 128, device=dev, generator=g), dim=-1).bfloat16()


def timed_block(corpus, Q, calls):
    L = _cabi.lib()
    L.flmr_scan_kernel_stats(None, None, 1)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(calls):
        s, p = R.maxsim_topk(corpus, Q, TOPK)
    b.record()
    torch.cuda.synchronize()
    tot, n = C.c_double(0), C.c_int64(0)
    L.flmr_scan_kernel_stats(C.byref(tot), C.byref(n), 1)
    return a.elapsed_time(b) / calls, tot.value / max(1, n.value), n.value // calls, s, p


def part1(n_passages, nbits, dev, blocks, calls):
    codes, residuals, cent, w, dl = synth(n_passages, nbits, seed=nbits, dev=dev)
    dec = decoded_corpus(codes, residuals, cent, w, nbits, dl, dev)
    cmp = compressed_corpus(codes, residuals, cent, w, nbits, dl, dev)
    del codes, residuals
    torch.cuda.empty_cache()
    total = torch.cuda.get_device_properties(dev).total_memory
    rows = int(cmp.info.n_rows)
    dec_bytes = int(dec.info.hbm_bytes) + (rows * 256 if dec.info.adopted else 0)
    res = {"nbits": nbits, "n_passages": n_passages, "tokens_per_passage": ND, "n_centroids": K_CENT,
           # an adopted token matrix is the caller's buffer and not in hbm_bytes: count it here
           "resident_hbm_bytes": {"decoded": dec_bytes, "compressed": int(cmp.info.hbm_bytes)},
           "algorithmic_bytes_per_corpus_pass": {
               "decoded": rows * 256,
               "compressed_hbm_stream": rows * (8 + 16 * nbits),
               "compressed_centroid_row_gathers": rows * 512,
               "centroid_table_bytes": K_CENT * 512},
           "passages_per_gpu": {k: passages_per_gpu(v / n_passages, rows / n_passages, total) for k, v in
                                (("decoded", dec_bytes), ("compressed", cmp.info.hbm_bytes))},
           "shapes": []}
    for nq, B in ((320, 16), (320, 1), (32, 16)):
        Q = queries(B, nq, seed=nq + B, dev=dev)
        for c in (dec, cmp):                 # warm-up of both paths at this shape
            timed_block(c, Q, 2)
        rows_t = {"decoded": [], "compressed": []}
        for blk in range(blocks):
            order = (("decoded", dec), ("compressed", cmp)) if blk % 2 == 0 else (("compressed", cmp), ("decoded", dec))
            out = {}
            for name, c in order:
                call_ms, scan_ms, launches, s, p = timed_block(c, Q, calls)
                rows_t[name].append((call_ms, scan_ms, launches))
                out[name] = (s, p)
            assert torch.equal(out["decoded"][0], out["compressed"][0]), (nbits, nq, B, blk)
            assert torch.equal(out["decoded"][1], out["compressed"][1]), (nbits, nq, B, blk)
        entry = {"nq": nq, "B": B, "k": TOPK, "blocks": blocks, "calls_per_block": calls, "topk_identical": True}
        for name, v in rows_t.items():
            call = np.array([x[0] for x in v])
            scan = np.array([x[1] for x in v])
            entry[name] = {"ms_per_scan_launch_median": float(np.median(scan)),
                           "ms_per_scan_launch_range": [float(scan.min()), float(scan.max())],
                           "scan_launches_per_call": int(v[0][2]),
                           "ms_per_call_median": float(np.median(call)),
                           "queries_per_s": float(B / (np.median(call) / 1e3))}
        entry["compressed_over_decoded_scan_time"] = (entry["compressed"]["ms_per_scan_launch_median"] /
                                                      entry["decoded"]["ms_per_scan_launch_median"])
        res["shapes"].append(entry)
        print(json.dumps(entry), flush=True)
    dec.close()
    cmp.close()
    torch.cuda.empty_cache()
    return res


def part2(n_passages, dev, slice_passages=1_000_000):
    nbits = 2
    g = torch.Generator(device=dev).manual_seed(99)
    cent = torch.nn.functional.normalize(torch.randn(K_CENT, 128, device=dev, generator=g), dim=-1).half().float()
    w = (torch.sort(torch.randn(1 << nbits, device=dev, generator=g)).values * 0.05).contiguous()
    dl = np.full(n_passages, ND, dtype=np.int32)
    slices = [(p0, min(n_passages, p0 + slice_passages)) for p0 in range(0, n_passages, slice_passages)]
    torch.cuda.synchronize()
    free0, total = torch.cuda.mem_get_info(dev)
    t0 = time.perf_counter()
    L = _cabi.lib()
    peak_used = 0
    b = _builder_from(cent, w, nbits, dl, dev, 0)
    for i, (p0, p1) in enumerate(slices):
        codes, residuals = synth_rows((p1 - p0) * ND, nbits, 1000 + i, dev)
        _append(b, codes, residuals)
        peak_used = max(peak_used, free0 - torch.cuda.mem_get_info(dev)[0])
        del codes, residuals
        torch.cuda.empty_cache()
    handle = C.c_void_p()
    _cabi.check(L.flmr_corpus_plaid_builder_finish(b, C.byref(handle)))
    cmp = R.FlatCorpus._from_handle(handle, dl, dev, 0, nbits=nbits)
    t_create = time.perf_counter() - t0
    Q = queries(16, 320, seed=5, dev=dev)
    timed_block(cmp, Q, 1)
    call_ms, scan_ms, launches, cs, cp = timed_block(cmp, Q, 3)
    info = {"n_passages": n_passages, "nbits": nbits, "stored_rows": int(cmp.info.n_rows),
            "row_limit_per_handle": MAX_SHARD_ROWS, "resident_hbm_bytes": int(cmp.info.hbm_bytes),
            "decoded_bytes_would_be": int(cmp.info.n_rows) * 256, "device_total_bytes": int(total),
            "peak_device_bytes_used_by_load": int(peak_used),
            "peak_over_resident": peak_used / cmp.info.hbm_bytes, "load_seconds": t_create,
            "B": 16, "nq": 320, "k": TOPK, "ms_per_call": call_ms, "ms_per_scan_launch": scan_ms}
    cmp.close()
    torch.cuda.empty_cache()
    lists_s, lists_p = [], []
    for i, (p0, p1) in enumerate(slices):
        codes, residuals = synth_rows((p1 - p0) * ND, nbits, 1000 + i, dev)
        dec = decoded_corpus(codes, residuals, cent, w, nbits, dl[p0:p1], dev, pid_base=p0)
        del codes, residuals
        s, p = R.maxsim_topk(dec, Q, TOPK)
        lists_s.append(s)
        lists_p.append(p)
        dec.close()
        torch.cuda.empty_cache()
    ms, mp = R.topk_merge(torch.stack(lists_s), torch.stack(lists_p), TOPK)
    assert torch.equal(ms, cs) and torch.equal(mp, cp), "capacity run: compressed top-k != merged decoded slices"
    info["topk_equals_merged_decoded_slices"] = True
    info["decoded_slices"] = len(lists_s)
    print(json.dumps(info), flush=True)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passages", type=int, default=1_000_000)
    ap.add_argument("--capacity-passages", type=int, default=11_000_000)
    ap.add_argument("--blocks", type=int, default=6)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("this probe measures the GPU; no CUDA device found")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _cabi.lib().flmr_set_profiling(1)
    report = {"card_before": card(), "part1": [], "part2": None}
    for nbits in (2, 8):
        report["part1"].append(part1(a.passages, nbits, dev, a.blocks, a.calls))
    if a.capacity_passages:
        report["part2"] = part2(a.capacity_passages, dev)
    report["card_after"] = card()
    text = json.dumps(report, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
