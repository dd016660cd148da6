"""Reader for the reference's PLAID index directories (SURVEY.md Appendix C; written by
third_party/ColBERT/colbert/indexing/collection_indexer.py + index_saver.py + codecs/residual.py)
and GPU decode into the flat bf16 store the scan kernel streams (SURVEY.md 8f-3), so a user of the
reference can switch without re-encoding the collection.

Only what the exhaustive scan needs is read: ``metadata.json`` (nbits, dim, num_chunks),
``centroids.pt``, ``buckets.pt``, ``<c>.codes.pt``, ``<c>.residuals.pt``, ``doclens.<c>.json``.
The IVF (``ivf.pid.pt``) and ``avg_residual.pt`` only serve PLAID's candidate generation / pruning.
"""
from __future__ import annotations

import ctypes as C
import json
import os
from typing import Optional, Tuple

import numpy as np
import torch

from . import _cabi


def read_plaid_metadata(path: str) -> dict:
    with open(os.path.join(path, "metadata.json")) as f:
        meta = json.load(f)
    cfg = meta["config"]
    return {"nbits": int(cfg["nbits"]), "dim": int(cfg["dim"]), "num_chunks": int(meta["num_chunks"]),
            "num_embeddings": int(meta.get("num_embeddings", -1))}


def decode_chunk(codes: torch.Tensor, residuals: torch.Tensor, centroids: torch.Tensor,
                 bucket_weights: torch.Tensor, nbits: int, out: torch.Tensor, normalize: bool = True) -> None:
    """GPU decode of one chunk into ``out`` (bf16 ``[n, 128]`` CUDA, may be a slice of the corpus matrix)."""
    dev = out.device
    codes = codes.to(dev, torch.int32).contiguous()
    residuals = residuals.to(dev, torch.uint8).contiguous()
    n = codes.numel()
    if residuals.shape != (n, _cabi.DIM * nbits // 8) or out.shape != (n, _cabi.DIM) or out.dtype != torch.bfloat16:
        raise ValueError("shape mismatch: codes %s residuals %s out %s" % (tuple(codes.shape),
                         tuple(residuals.shape), tuple(out.shape)))
    if not out.is_contiguous():
        raise ValueError("out must be contiguous")
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().flmr_plaid_decode(
            C.c_void_p(codes.data_ptr()), C.c_void_p(residuals.data_ptr()), n,
            C.c_void_p(centroids.data_ptr()), centroids.size(0), C.c_void_p(bucket_weights.data_ptr()),
            nbits, _cabi.DIM, int(normalize), C.c_void_p(out.data_ptr()), int(dev.index),
            C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))


def read_plaid_doclens(path: str, num_chunks: int):
    """Per-chunk passage lengths (``doclens.<c>.json``, index_saver.py:83-85)."""
    out = []
    for c in range(num_chunks):
        with open(os.path.join(path, "doclens.%d.json" % c)) as f:
            out.append(np.asarray(json.load(f), dtype=np.int64))
    return out


def _shard_pieces(chunk_doclens, p0: int, p1: int):
    """The chunks that hold passages ``[p0, p1)``: (chunk, first token row, one-past-last row, doclens slice,
    tokens in the chunk) each."""
    pieces, c0 = [], 0
    for c, dl in enumerate(chunk_doclens):
        a, b = max(p0, c0) - c0, min(p1, c0 + len(dl)) - c0
        if a < b:
            off = np.concatenate([[0], np.cumsum(dl)])
            pieces.append((c, int(off[a]), int(off[b]), dl[a:b], int(off[-1])))
        c0 += len(dl)
    return pieces


# ---- compressed residency ---------------------------------------------------------------------------------------
# A shard is decoded into bf16 (256 B per token) when that fits the device; otherwise it stays compressed
# (4 + 16 * nbits + 4 B per token: code, packed residual, inverse norm) and the scan kernel decodes it.
DECODE_MARGIN_BYTES = 4 << 30    # HBM left free beside a decoded shard: workspaces, query batches, score rows
DECODE_MARGIN_FRACTION = 0.10    # ... or this share of the free memory, whichever is larger
MAX_SHARD_ROWS = (1 << 31) - 1 - _cabi.TILE_TOKENS   # stored (padded) rows one corpus handle can hold, either way

_residency_override = "auto"


def debug_set_residency(mode: str) -> None:
    """Test infrastructure: how ``FlatCorpus.from_plaid`` holds a PLAID shard on this process — ``"auto"`` (the
    product behaviour, :func:`keep_compressed`), ``"decoded"`` or ``"compressed"`` — so tests can hold either
    path against the other on indexes of any size."""
    global _residency_override
    if mode not in ("auto", "decoded", "compressed"):
        raise ValueError("mode must be 'auto', 'decoded' or 'compressed', got %r" % (mode,))
    _residency_override = mode


def decoded_shard_bytes(doclens) -> int:
    """HBM a decoded shard takes: the bf16 token matrix, plus its padded copy when some passage length is not a
    multiple of 4 (the corpus then cannot adopt the decoded matrix)."""
    dl = np.asarray(doclens, dtype=np.int64)
    n_tokens = int(dl.sum())
    rows = int(((dl + _cabi.TOKEN_GROUP - 1) // _cabi.TOKEN_GROUP * _cabi.TOKEN_GROUP).sum())
    return _cabi.DIM * 2 * (n_tokens + (rows if rows != n_tokens else 0))


def keep_compressed(decoded_bytes: int, free_bytes: int) -> bool:
    """The residency rule: keep the shard compressed when its decoded size does not fit the device's free memory
    after a margin of max(DECODE_MARGIN_BYTES, DECODE_MARGIN_FRACTION * free)."""
    margin = max(DECODE_MARGIN_BYTES, int(DECODE_MARGIN_FRACTION * free_bytes))
    return decoded_bytes > free_bytes - margin


def use_compressed(doclens, device) -> bool:
    """What ``FlatCorpus.from_plaid`` does for a shard with these doclens on ``device``."""
    if _residency_override != "auto":
        return _residency_override == "compressed"
    free, _total = torch.cuda.mem_get_info(device)
    return keep_compressed(decoded_shard_bytes(doclens), free)


def plaid_to_compressed(path: str, device=None, passage_range: Optional[Tuple[int, int]] = None):
    """Load a PLAID index — all of it, or the passages ``[p0, p1)`` only (only the chunks that overlap are read) —
    as a compressed corpus handle: (handle, doclens int32, nbits).  Chunk by chunk through
    ``flmr_corpus_plaid_builder_*``: the device holds the handle's arrays plus ONE chunk's codes and residuals at a
    time, and the chunk staging is handed back to the driver before returning."""
    if not torch.cuda.is_available():
        raise RuntimeError("the compressed PLAID corpus lives on the GPU; there is no CPU fallback")
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    meta = read_plaid_metadata(path)
    if meta["dim"] != _cabi.DIM:
        raise ValueError("dim=%d (only %d is supported)" % (meta["dim"], _cabi.DIM))
    nbits = meta["nbits"]
    chunk_doclens = read_plaid_doclens(path, meta["num_chunks"])
    n_total = int(sum(len(d) for d in chunk_doclens))
    p0, p1 = (0, n_total) if passage_range is None else passage_range
    if not 0 <= p0 < p1 <= n_total:
        raise ValueError("passage_range %s outside [0, %d] or empty" % (passage_range, n_total))
    pieces = _shard_pieces(chunk_doclens, p0, p1)
    doclens = np.ascontiguousarray(np.concatenate([p[3] for p in pieces]), dtype=np.int32)
    packed = _cabi.DIM * nbits // 8
    L = _cabi.lib()

    def chunk(c, r0, r1, n_chunk):
        cc = torch.load(os.path.join(path, "%d.codes.pt" % c), map_location="cpu")
        rr = torch.load(os.path.join(path, "%d.residuals.pt" % c), map_location="cpu")
        if cc.numel() != n_chunk:
            raise ValueError("chunk %d holds %d codes but its doclens sum to %d" % (c, cc.numel(), n_chunk))
        if tuple(rr.shape) != (n_chunk, packed):
            raise ValueError("chunk %d residuals have shape %s, expected (%d, %d)" % (c, tuple(rr.shape), n_chunk,
                                                                                     packed))
        return cc[r0:r1].to(torch.int32), rr[r0:r1].to(torch.uint8)

    with torch.cuda.device(device):
        b = _plaid_builder(path, nbits, doclens, device, p0)
        try:
            for c, r0, r1, _, n_chunk in pieces:
                codes, residuals = chunk(c, r0, r1, n_chunk)
                _append(b, codes.to(device), residuals.to(device))
                del codes, residuals
            handle = C.c_void_p()
            _cabi.check(L.flmr_corpus_plaid_builder_finish(b, C.byref(handle)))
            b = None
        finally:
            if b is not None:
                L.flmr_corpus_plaid_builder_destroy(b)
            torch.cuda.empty_cache()     # the chunk staging goes back to the driver, not to torch's cache
    return handle, doclens, nbits


def _plaid_builder(path, nbits, doclens, device, pid_base):
    centroids = torch.load(os.path.join(path, "centroids.pt"), map_location="cpu").float().to(device).contiguous()
    _cutoffs, weights = torch.load(os.path.join(path, "buckets.pt"), map_location="cpu")
    return _builder_from(centroids, weights.float().to(device).contiguous(), nbits, doclens, device, pid_base)


def _builder_from(centroids, bucket_weights, nbits, doclens, device, pid_base) -> C.c_void_p:
    dl = np.ascontiguousarray(np.asarray(doclens), dtype=np.int32)
    b = C.c_void_p()
    torch.cuda.current_stream(device).synchronize()   # the copies that filled the centroids are done
    _cabi.check(_cabi.lib().flmr_corpus_plaid_builder_create(
        C.c_void_p(centroids.data_ptr()), centroids.size(0), C.c_void_p(bucket_weights.data_ptr()), int(nbits),
        dl.ctypes.data_as(C.c_void_p), len(dl), _cabi.DIM, int(torch.device(device).index), int(pid_base),
        C.byref(b)))
    return b


def _append(b, codes: torch.Tensor, residuals: torch.Tensor) -> None:
    codes, residuals = codes.contiguous(), residuals.contiguous()
    torch.cuda.current_stream(codes.device).synchronize()   # the chunk's copies to the device are done
    _cabi.check(_cabi.lib().flmr_corpus_plaid_builder_append(
        b, C.c_void_p(codes.data_ptr()), C.c_void_p(residuals.data_ptr()), codes.numel()))


def create_compressed(codes: torch.Tensor, residuals: torch.Tensor, centroids: torch.Tensor,
                      bucket_weights: torch.Tensor, nbits: int, doclens, device, pid_base: int = 0,
                      chunk_passages: Optional[int] = None) -> C.c_void_p:
    """A compressed corpus handle from CUDA tensors of ``device`` (codes int32 ``[n_tokens]``, residuals uint8
    ``[n_tokens, 16 * nbits]``, centroids and bucket weights fp32), packed ``chunk_passages`` passages at a time
    (all at once by default)."""
    dl = np.ascontiguousarray(np.asarray(doclens), dtype=np.int32)
    L = _cabi.lib()
    with torch.cuda.device(device):
        b = _builder_from(centroids, bucket_weights, nbits, dl, device, pid_base)
        try:
            off = np.concatenate([[0], np.cumsum(dl, dtype=np.int64)])
            step = len(dl) if chunk_passages is None else int(chunk_passages)
            for a in range(0, len(dl), step):
                r0, r1 = int(off[a]), int(off[min(len(dl), a + step)])
                _append(b, codes[r0:r1], residuals[r0:r1])
            handle = C.c_void_p()
            _cabi.check(L.flmr_corpus_plaid_builder_finish(b, C.byref(handle)))
            b = None
        finally:
            if b is not None:
                L.flmr_corpus_plaid_builder_destroy(b)
    return handle


def plaid_to_flat(path: str, device=None, passage_range: Optional[Tuple[int, int]] = None
                  ) -> Tuple[torch.Tensor, np.ndarray]:
    """Decode a PLAID index — all of it, or the passages ``[p0, p1)`` only (one GPU's shard: only the chunks
    that overlap are read) — into (tokens bf16 ``[n_tokens, 128]`` on the GPU, doclens int32)."""
    if not torch.cuda.is_available():
        raise RuntimeError("PLAID decode runs on the GPU; there is no CPU fallback")
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    meta = read_plaid_metadata(path)
    if meta["dim"] != _cabi.DIM:
        raise ValueError("dim=%d (only %d is supported)" % (meta["dim"], _cabi.DIM))
    centroids = torch.load(os.path.join(path, "centroids.pt"), map_location="cpu").float().to(device).contiguous()
    _cutoffs, weights = torch.load(os.path.join(path, "buckets.pt"), map_location="cpu")
    weights = weights.float().to(device).contiguous()
    chunk_doclens = read_plaid_doclens(path, meta["num_chunks"])
    n_total = int(sum(len(d) for d in chunk_doclens))
    p0, p1 = (0, n_total) if passage_range is None else passage_range
    if not 0 <= p0 <= p1 <= n_total:
        raise ValueError("passage_range %s outside [0, %d]" % (passage_range, n_total))
    pieces = _shard_pieces(chunk_doclens, p0, p1)
    tokens = torch.empty((sum(p[2] - p[1] for p in pieces), _cabi.DIM), dtype=torch.bfloat16, device=device)
    row = 0
    for c, r0, r1, _, n_chunk in pieces:
        codes = torch.load(os.path.join(path, "%d.codes.pt" % c), map_location="cpu")
        residuals = torch.load(os.path.join(path, "%d.residuals.pt" % c), map_location="cpu")
        if codes.numel() != n_chunk:
            raise ValueError("chunk %d holds %d codes but its doclens sum to %d" % (c, codes.numel(), n_chunk))
        decode_chunk(codes[r0:r1], residuals[r0:r1], centroids, weights, meta["nbits"], tokens[row:row + r1 - r0])
        row += r1 - r0
    doclens = np.concatenate([p[3] for p in pieces]) if pieces else np.empty(0, dtype=np.int64)
    return tokens, doclens.astype(np.int32)
