"""Index-load throughput (GPU box): write a synthetic flat index of `--gigabytes` to `--dir` (chunks of 25k
passages, as the Indexer writes them), evict its files from the page cache, and time FlatCorpus.from_index —
the C-level streaming builder (pread into two pinned buffers with 8 threads, overlapped H2D, padded layout).

    python tools/index_load_probe.py --gigabytes 8 --dir /dev/shm/flmr_idx
"""
import argparse
import os
import shutil
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gigabytes", type=float, default=8.0)
    ap.add_argument("--nd", type=int, default=180)
    ap.add_argument("--dir", default="/tmp/flmr_idx_probe")
    ap.add_argument("--ragged", action="store_true")
    args = ap.parse_args()
    import numpy as np
    import torch
    import ravqa_b200 as R
    from ravqa_b200.index_io import finalize_chunked_index, save_flat_chunk
    n = int(args.gigabytes * 1e9 / (args.nd * 256))
    shutil.rmtree(args.dir, ignore_errors=True)
    g = torch.Generator(device="cuda").manual_seed(0)
    t0 = time.perf_counter()
    c, p = 0, 0
    while p < n:
        m = min(25_000, n - p)
        dl = (np.random.default_rng(c).integers(args.nd // 2, args.nd + 1, size=m) if args.ragged
              else np.full(m, args.nd)).astype(np.int32)
        x = torch.nn.functional.normalize(torch.randn((int(dl.sum()), 128), device="cuda", generator=g), dim=-1)
        save_flat_chunk(args.dir, c, p, x.to(torch.bfloat16).cpu(), dl)
        p += m
        c += 1
    finalize_chunked_index(args.dir, c)
    t_write = time.perf_counter() - t0
    size = sum(os.path.getsize(os.path.join(args.dir, f)) for f in os.listdir(args.dir)) / 1e9
    print("wrote %.2f GB in %d chunks to %s (%.1f s)" % (size, c, args.dir, t_write), flush=True)
    # evict only this index's own pages (a per-file hint; clean pages of these files are dropped)
    cold = False
    try:
        for f in os.listdir(args.dir):
            fd = os.open(os.path.join(args.dir, f), os.O_RDONLY)
            try:
                os.fsync(fd)
                os.posix_fadvise(fd, 0, 0, os.POSIX_FADV_DONTNEED)
            finally:
                os.close(fd)
        cold = True
    except (OSError, AttributeError):
        pass
    for attempt in ("cold" if cold else "page-cache", "page-cache"):
        torch.cuda.synchronize()
        corpus = R.FlatCorpus.from_index(args.dir)
        s = corpus.load_stats
        print("load (%s): %.2f GB in %.2f s = %.2f GB/s (host fill %.2f s; %d passages, adopted=%d) -> 46.08 GB in %.1f s"
              % (attempt, s["gigabytes"], s["seconds"], s["gb_per_s"], s["host_fill_seconds"], corpus.n_passages,
                 corpus.info.adopted, 46.08 / s["gb_per_s"]), flush=True)
        corpus.close()
    # the path it replaces: numpy read of the shard + pageable cudaMemcpy in flmr_corpus_create
    from ravqa_b200.index_io import load_flat_index
    t0 = time.perf_counter()
    tokens, doclens, _ = load_flat_index(args.dir)
    corpus = R.FlatCorpus(tokens, doclens)
    dt = time.perf_counter() - t0
    print("round-1 path (load_flat_index -> FlatCorpus): %.2f s = %.2f GB/s" % (dt, size / dt), flush=True)
    corpus.close()
    shutil.rmtree(args.dir, ignore_errors=True)


if __name__ == "__main__":
    main()
