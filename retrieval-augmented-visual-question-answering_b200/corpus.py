"""Resident passage-token corpus shard (replaces the PLAID index residency of the reference:
``IndexScorer.__init__`` / ``IndexLoader``, third_party/ColBERT/colbert/search/index_storage.py:21-66,
index_loader.py:13-86).

The reference keeps centroids + residual codes + an IVF and decompresses ~256 survivors per query;
here the whole shard is a flat bf16 ``[sum(doclens), 128]`` matrix in HBM plus ``doclens`` — exactly
the ``(D_packed, D_lengths)`` operand pair of ``colbert_score_packed`` (colbert/modeling/colbert.py:289)
— scanned exhaustively by the fused kernel.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Union

import numpy as np
import torch

from . import _cabi


def _as_doclens(doclens) -> np.ndarray:
    if isinstance(doclens, torch.Tensor):
        doclens = doclens.detach().cpu().numpy()
    arr = np.ascontiguousarray(np.asarray(doclens), dtype=np.int32)
    if arr.ndim != 1:
        raise ValueError("doclens must be 1-D")
    return arr


class FlatCorpus:
    """One GPU's shard of the passage-token matrix, resident in HBM.

    tokens   : ``[sum(doclens), 128]`` tensor (bf16 preferred; fp16/fp32 are rounded to bf16), on CPU
               or on the target GPU.  A CUDA bf16 tensor whose doclens are all multiples of 4 is
               adopted zero-copy (and kept alive by this object).
    doclens  : per-passage token counts (>= 1 each).
    pid_base : global id of this shard's first passage (sharded search, SURVEY.md §8e).
    """

    def __init__(self, tokens: torch.Tensor, doclens, device: Optional[Union[int, torch.device]] = None,
                 pid_base: int = 0, adopt: bool = True):
        if not torch.cuda.is_available():
            raise RuntimeError("FlatCorpus needs a CUDA device: there is no CPU fallback for this path")
        L = _cabi.lib()
        self.doclens = _as_doclens(doclens)
        if tokens.dim() != 2 or tokens.size(1) != _cabi.DIM:
            raise ValueError("tokens must be [sum(doclens), %d], got %s" % (_cabi.DIM, tuple(tokens.shape)))
        if int(self.doclens.sum()) != tokens.size(0):
            raise ValueError("sum(doclens)=%d != tokens rows=%d" % (int(self.doclens.sum()), tokens.size(0)))
        if device is None:
            device = tokens.device if tokens.is_cuda else torch.device("cuda", torch.cuda.current_device())
        device = torch.device(device) if not isinstance(device, torch.device) else device
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device
        tokens = tokens.detach()
        if tokens.dtype != torch.bfloat16:
            tokens = tokens.to(torch.bfloat16)
        tokens = tokens.contiguous()
        if tokens.is_cuda and tokens.device != device:
            tokens = tokens.to(device)
        flags = _cabi.CORPUS_ADOPT if (adopt and tokens.is_cuda) else _cabi.CORPUS_COPY
        if tokens.is_cuda:
            torch.cuda.current_stream(device).synchronize()  # producer kernels of `tokens` are done
        handle = C.c_void_p()
        _cabi.check(L.flmr_corpus_create(C.c_void_p(tokens.data_ptr()),
                                         self.doclens.ctypes.data_as(C.c_void_p),
                                         int(self.doclens.shape[0]), _cabi.DIM, int(device.index),
                                         int(pid_base), flags, C.byref(handle)))
        self._h = handle
        info = _cabi.CorpusInfo()
        _cabi.check(L.flmr_corpus_info(self._h, C.byref(info)))
        self.info = info
        self._keepalive = tokens if info.adopted else None
        self._ws = None
        self.pid_base = int(pid_base)
        self.load_stats = None
        self.nbits = 0

    @classmethod
    def _from_handle(cls, handle, doclens: np.ndarray, device: torch.device, pid_base: int,
                     nbits: int = 0) -> "FlatCorpus":
        self = cls.__new__(cls)
        self.doclens = doclens
        self.device = device
        self._h = handle
        info = _cabi.CorpusInfo()
        _cabi.check(_cabi.lib().flmr_corpus_info(self._h, C.byref(info)))
        self.info = info
        self._keepalive = None
        self._ws = None
        self.pid_base = int(pid_base)
        self.load_stats = None
        self.nbits = int(nbits)      # != 0: the handle came from flmr_corpus_create_plaid / the PLAID builder
        return self

    @classmethod
    def from_index(cls, path: str, device=None, rank: int = 0, world_size: int = 1) -> "FlatCorpus":
        """Load a flat index (index_io.py) — or, with world_size > 1, only this rank's contiguous,
        token-balanced passage shard of it (SURVEY.md 8e) — into HBM.

        The token files are streamed by the C-level corpus builder: ``pread`` straight into two pinned staging
        buffers (8 reader threads, the fill of one buffer overlaps the DMA of the other) and from there into the
        padded layout — no numpy copy of the shard, no pageable ``cudaMemcpy``.  ``load_stats`` records seconds
        and GB/s (replaces IndexLoader / ResidualEmbeddings.load_chunks, colbert/search/index_loader.py:24-62)."""
        import time
        from .index_io import index_token_files
        from .sharded import shard_ranges
        if not torch.cuda.is_available():
            raise RuntimeError("FlatCorpus needs a CUDA device: there is no CPU fallback for this path")
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        device = torch.device(device) if not isinstance(device, torch.device) else device
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        all_doclens, files = index_token_files(path)        # files: [(path, first passage, n passages, n rows)]
        p0, p1 = shard_ranges(all_doclens, world_size)[rank] if world_size > 1 else (0, len(all_doclens))
        if p0 == p1:
            return None          # more ranks than passages: this rank holds nothing (Searcher copes)
        doclens = np.ascontiguousarray(all_doclens[p0:p1], dtype=np.int32)
        L = _cabi.lib()
        t0 = time.perf_counter()
        b = C.c_void_p()
        _cabi.check(L.flmr_corpus_builder_create(doclens.ctypes.data_as(C.c_void_p), len(doclens), _cabi.DIM,
                                                 int(device.index), int(p0), C.byref(b)))
        try:
            for fname, f0, fn, _rows in files:
                a, e = max(p0, f0), min(p1, f0 + fn)
                if a >= e:
                    continue
                row_a = int(all_doclens[f0:a].sum())
                rows = int(all_doclens[a:e].sum())
                _cabi.check(L.flmr_corpus_builder_append_file(b, fname.encode(), row_a * _cabi.DIM * 2, rows))
            handle, fill_s = C.c_void_p(), C.c_double(0)
            _cabi.check(L.flmr_corpus_builder_finish(b, C.byref(handle), C.byref(fill_s)))
            b = None
        finally:
            if b is not None:
                L.flmr_corpus_builder_destroy(b)
        self = cls._from_handle(handle, doclens, device, p0)
        dt = time.perf_counter() - t0
        gb = float(doclens.sum()) * _cabi.DIM * 2 / 1e9
        self.load_stats = {"seconds": dt, "gigabytes": gb, "gb_per_s": gb / dt, "host_fill_seconds": fill_s.value,
                           "rank": rank, "world_size": world_size}
        return self

    @classmethod
    def from_plaid(cls, path: str, device=None, rank: int = 0, world_size: int = 1) -> "FlatCorpus":
        """Load a reference PLAID index directory (plaid.py) and keep it resident — with world_size > 1 only
        this rank's contiguous, token-balanced passage shard (SURVEY.md 8e).  The shard is decoded into bf16 on
        the GPU when that fits the device's free memory (plaid.keep_compressed); otherwise it stays compressed in
        HBM and the scan decodes it on the fly.  Either way searches return the same bits."""
        from .plaid import plaid_to_compressed, plaid_to_flat, read_plaid_doclens, read_plaid_metadata, use_compressed
        from .sharded import shard_ranges
        if not torch.cuda.is_available():
            raise RuntimeError("FlatCorpus needs a CUDA device: there is no CPU fallback for this path")
        all_doclens = np.concatenate(read_plaid_doclens(path, read_plaid_metadata(path)["num_chunks"]))
        p0, p1 = shard_ranges(all_doclens, world_size)[rank] if world_size > 1 else (0, len(all_doclens))
        if p0 == p1:
            return None
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        if use_compressed(all_doclens[p0:p1], dev):
            handle, doclens, nbits = plaid_to_compressed(path, dev, passage_range=(p0, p1))
            return cls._from_handle(handle, doclens, dev, p0, nbits=nbits)
        tokens, doclens = plaid_to_flat(path, dev, passage_range=(p0, p1))
        return cls(tokens, doclens, device=tokens.device, pid_base=p0)

    @classmethod
    def from_plaid_arrays(cls, codes: torch.Tensor, residuals: torch.Tensor, centroids: torch.Tensor,
                          bucket_weights: torch.Tensor, nbits: int, doclens, device=None, pid_base: int = 0,
                          chunk_passages: Optional[int] = None) -> "FlatCorpus":
        """A compressed shard from PLAID arrays already on the GPU (codes int32, residuals uint8, centroids and
        bucket weights fp32; see plaid.create_compressed)."""
        from .plaid import create_compressed
        dev = codes.device if device is None else torch.device(device)
        dl = _as_doclens(doclens)
        handle = create_compressed(codes, residuals, centroids, bucket_weights, nbits, dl, dev, pid_base,
                                   chunk_passages=chunk_passages)
        return cls._from_handle(handle, dl, dev, pid_base, nbits=nbits)

    # -- properties ---------------------------------------------------------------------------
    @property
    def n_passages(self) -> int:
        return int(self.info.n_passages)

    @property
    def n_tokens(self) -> int:
        return int(self.info.n_tokens)

    @property
    def compressed(self) -> bool:
        """True when the shard is held as PLAID codes + residuals (``nbits`` per dim) and decoded by the scan."""
        return self.nbits != 0

    @property
    def handle(self) -> C.c_void_p:
        if self._h is None:
            raise RuntimeError("corpus was closed")
        return self._h

    def workspace(self) -> C.c_void_p:
        """Default per-corpus scratch (single-threaded use, like the reference Searcher)."""
        if self._ws is None:
            ws = C.c_void_p()
            _cabi.check(_cabi.lib().flmr_workspace_create(self.handle, 64, 1024, C.byref(ws)))
            self._ws = ws
        return self._ws

    def gather_padded(self, pids: torch.Tensor, nd_max: Optional[int] = None):
        """Retrieved passages as a padded batch, straight out of HBM: ``pids`` (any shape, global ids) ->
        (tokens bf16 ``[*pids.shape, nd_max, 128]``, mask bool ``[*pids.shape, nd_max, 1]``).  ``nd_max``
        defaults to the longest requested passage.  Ids outside this shard give an all-masked zero row.
        Replaces the host-dictionary lookup + stack + H2D of rag_model_blip.py:414-425."""
        shape = tuple(pids.shape)
        flat = pids.detach().reshape(-1).to(device=self.device, dtype=torch.int64).contiguous()
        if nd_max is None:
            local = (flat - self.pid_base).clamp(0, self.n_passages - 1).cpu().numpy()
            nd_max = int(self.doclens[local].max()) if flat.numel() else 1
        out = torch.empty((flat.numel(), nd_max, _cabi.DIM), dtype=torch.bfloat16, device=self.device)
        mask = torch.empty((flat.numel(), nd_max), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _cabi.check(_cabi.lib().flmr_corpus_gather(
                self.handle, C.c_void_p(flat.data_ptr()), flat.numel(), int(nd_max), C.c_void_p(out.data_ptr()),
                C.c_void_p(mask.data_ptr()), C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        return out.view(*shape, nd_max, _cabi.DIM), mask.bool().view(*shape, nd_max, 1)

    def close(self) -> None:
        L = _cabi.lib()
        if self._ws is not None:
            L.flmr_workspace_destroy(self._ws)
            self._ws = None
        if self._h is not None:
            torch.cuda.synchronize(self.device)
            L.flmr_corpus_destroy(self._h)
            self._h = None
        self._keepalive = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __repr__(self) -> str:
        i = self.info
        return ("FlatCorpus(n_passages=%d, n_tokens=%d, device=%s, pid_base=%d, n_ctas=%d, adopted=%d, nbits=%d)"
                % (i.n_passages, i.n_tokens, self.device, i.pid_base, i.n_ctas, i.adopted, self.nbits))
