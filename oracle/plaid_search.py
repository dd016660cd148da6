"""CPU restatement of the reference's PLAID search — the "FAISS+ColBERT path" the north star replaces.

TEST INFRASTRUCTURE.  Only tests/, tools/ probes and bench.py's CPU-baseline legs may import this
module; the product path (retrieval-augmented-visual-question-answering_b200/) never does.

What RA-VQA runs at evaluation time under DDP is ColBERT's PLAID pipeline on CPU
(src/executors/FLMR_executor.py:778-792 -> colbert/searcher.py:91-132 -> IndexScorer.rank).  This
module restates the Python glue of that pipeline and calls the reference's OWN native kernels,
compiled in place by oracle/build_ref.py into oracle/_ref/ (filter_pids_cpp, decompress_residuals_cpp,
segmented_lookup_cpp, segmented_maxsim_cpp).  Restatements of those four kernels are kept beside them
(filter_pids_np, decompress_residuals_restated, segmented_lookup_restated, maxsim_oracle.segmented_maxsim)
so the pruning rule is spelled out, and the search runs where the compiled kernels are absent.

Pinned by tests/test_plaid_search.py against tests/golden/plaid_search.npz, which was produced by the
reference's unmodified IndexScorer.rank / retrieve (tests/golden/make_golden_plaid_search.py).

Reference map (third_party/ColBERT/colbert/...):
    PlaidIndex.build     indexing/collection_indexer.py:290-314 (_compute_avg_residual: bucket cutoffs/weights)
                         indexing/codecs/residual.py:168-223 (compress / binarize / compress_into_codes)
                         indexing/collection_indexer.py:419-456 (_build_ivf) + indexing/utils.py:8-56 (optimize_ivf)
    PlaidIndex.load      search/index_loader.py:20-78, indexing/codecs/residual.py:128-150 (ResidualCodec.load)
    PlaidSearcher.get_cells / candidates
                         search/candidate_generation.py:11-20, 30-36, 45-62; search/strided_tensor.py:60-97
    PlaidSearcher.retrieve / rank / score_pids
                         search/index_storage.py:66-100, 102-182 (CPU branch)
    colbert_score_packed modeling/colbert.py:294-311
K-means itself (faiss in the reference, indexing/collection_indexer.py:236-262) is NOT restated: faiss is
absent from this image, so `train_centroids` is a seeded spherical Lloyd iteration and says so.
"""
from __future__ import annotations

import itertools
import json
import os

import numpy as np
import torch

from . import build_ref, maxsim_oracle

_EXT = {}


def _ext(name):
    """The compiled reference extension `name` (oracle/_ref/<name>.so); raises when it was never built."""
    if name not in _EXT:
        mod = build_ref.load(name)
        if mod is None:
            raise RuntimeError("oracle/_ref/%s.so is missing: run `python oracle/build_ref.py` in the build "
                               "container (needs /root/reference)" % name)
        _EXT[name] = mod
    return _EXT[name]


def have_reference_kernels() -> bool:
    return all(os.path.exists(build_ref.out_path(n)) for n in build_ref.SOURCES)


# ----------------------------------------------------------------------------------------------
# index
# ----------------------------------------------------------------------------------------------
def reversed_bit_map(nbits: int) -> torch.Tensor:
    """residual.py:49-71 — per byte, reverse the bit order inside every nbits-wide field."""
    out = []
    for byte in range(256):
        z = 0
        for field in range(8 // nbits):
            x = (byte >> (8 - nbits * (field + 1))) & ((1 << nbits) - 1)
            y = int(format(x, "0%db" % nbits)[::-1], 2)
            z = (z << nbits) | y
        out.append(z)
    return torch.tensor(out).to(torch.uint8)


def decompression_lookup_table(n_weights: int, nbits: int) -> torch.Tensor:
    """residual.py:73-88 — every ordered tuple of (8/nbits) bucket indices, one row per byte value."""
    return torch.tensor(list(itertools.product(range(n_weights), repeat=8 // nbits))).to(torch.uint8)


def train_centroids(sample: torch.Tensor, k: int, iters: int = 4, seed: int = 0, device=None) -> torch.Tensor:
    """Seeded spherical Lloyd k-means (stand-in for faiss.Kmeans, collection_indexer.py:236-262).

    Returns fp32 centroids rounded through fp16, as the reference stores them (residual.py:160)."""
    g = torch.Generator().manual_seed(seed)
    x = sample.float()
    c = x[torch.randperm(x.size(0), generator=g)[:k]].clone()
    if device is not None:
        x, c = x.to(device), c.to(device)
    for _ in range(iters):
        assign = torch.cat([(xb @ c.T).argmax(dim=1) for xb in x.split(1 << 16)])
        sums = torch.zeros_like(c).index_add_(0, assign, x)
        cnt = torch.bincount(assign, minlength=k).unsqueeze(1)
        c = torch.where(cnt > 0, torch.nn.functional.normalize(sums / cnt.clamp_min(1), dim=-1), c)
    return c.cpu().half().float()


class PlaidIndex:
    """In-memory PLAID index with exactly the tensors IndexScorer holds on CPU (index_storage.py:17-64)."""

    def __init__(self, centroids, bucket_cutoffs, bucket_weights, codes, residuals, doclens, ivf, ivf_lengths,
                 nbits, dim=128):
        self.dim, self.nbits = int(dim), int(nbits)
        self.centroids = centroids.float().contiguous()                       # residual.py:27 (CPU: fp32)
        self.bucket_cutoffs = bucket_cutoffs
        self.bucket_weights = bucket_weights.to(torch.float32).contiguous()   # residual.py:41-42
        self.codes = codes.to(torch.int32).contiguous()                        # residual_embeddings.py:25 (int32)
        self.residuals = residuals.to(torch.uint8).contiguous()
        self.doclens = torch.as_tensor(doclens).long().contiguous()            # index_loader.py:57
        zero = torch.zeros(1, dtype=torch.long)
        self.offsets = torch.cat((zero, torch.cumsum(self.doclens, dim=0)))    # strided_tensor_core.py:31-32
        self.ivf = ivf.contiguous()                                            # int32 pids, grouped by centroid
        self.ivf_lengths = ivf_lengths.long().contiguous()
        self.ivf_offsets = torch.cat((zero, torch.cumsum(self.ivf_lengths, dim=0)))
        self.reversed_bit_map = reversed_bit_map(self.nbits)
        self.lut = decompression_lookup_table(len(self.bucket_weights), self.nbits)
        # The reference pads strided tensors so a max-stride view never runs off the end
        # (strided_tensor_core.py:34-40); the CPU lookups below index by offset+length only, so no padding.

    # -- build ---------------------------------------------------------------------------------
    @staticmethod
    def compress_into_codes(centroids, embs):
        """residual.py:203-221: nearest centroid by inner product, in batches of 2^29 / K columns.
        Runs where `centroids` lives (the reference: fp32 on CPU, fp16 on CUDA; here always fp32)."""
        out = []
        for batch in embs.split((1 << 29) // centroids.size(0)):
            out.append((centroids @ batch.to(centroids.device).float().T).max(dim=0).indices)
        return torch.cat(out)

    @staticmethod
    def binarize(residuals, bucket_cutoffs, nbits):
        """residual.py:186-201: bucket index per dimension -> nbits bits, least significant first ->
        packed 8 per byte, first bit in the MSB (np.packbits order; done with integer weights so the same
        code runs on either device)."""
        dim = residuals.size(1)
        assert dim % 8 == 0 and dim % (nbits * 8) == 0, (dim, nbits)
        b = torch.bucketize(residuals.float(), bucket_cutoffs.to(residuals.device)).to(dtype=torch.uint8)
        bits = (b.unsqueeze(-1) >> torch.arange(0, nbits, dtype=torch.uint8, device=b.device)) & 1
        bits = bits.reshape(residuals.size(0), dim * nbits // 8, 8).to(torch.int32)
        weights = torch.tensor([128, 64, 32, 16, 8, 4, 2, 1], dtype=torch.int32, device=b.device)
        return (bits * weights).sum(dim=-1).to(torch.uint8)

    @classmethod
    def build(cls, embs, doclens, centroids, nbits, heldout=None, device=None):
        """Codec statistics + compression + IVF for `embs` [n_emb,128] (already L2-normalised).

        `heldout`: the sample bucket cutoffs/weights are estimated on (collection_indexer.py:290-314 uses
        the 5% held-out split of the k-means sample); defaults to (a bounded prefix of) `embs`.
        `device`: where the nearest-centroid matmuls and the bit packing run — index build is never
        inside a timed region; None = CPU, as the reference does without GPUs."""
        dev = torch.device("cpu") if device is None else torch.device(device)
        doclens = torch.as_tensor(doclens).long().cpu()
        K, n_p = centroids.size(0), doclens.numel()
        cent = centroids.float().to(dev)
        heldout = embs[: 1 << 17] if heldout is None else heldout
        heldout = heldout.to(dev).float()
        h_res = heldout - cent[cls.compress_into_codes(cent, heldout)]
        num_options = 2 ** nbits
        quantiles = (torch.arange(0, num_options) * (1 / num_options)).to(dev)
        flat = h_res.flatten()
        if flat.numel() > (1 << 24):                                          # torch.quantile's input limit
            flat = flat[torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[: 1 << 24].to(dev)]
        bucket_cutoffs = flat.quantile(quantiles[1:])
        bucket_weights = flat.quantile(quantiles + (0.5 / num_options))
        codes, residuals = [], []
        for batch in embs.split(1 << 18):                                     # residual.py:168-184
            batch = batch.to(dev).float()
            c = cls.compress_into_codes(cent, batch)
            codes.append(c.cpu())
            residuals.append(cls.binarize(batch - cent[c], bucket_cutoffs, nbits).cpu())
        codes, residuals = torch.cat(codes), torch.cat(residuals)
        # _build_ivf (collection_indexer.py:433-445): embedding ids sorted by code + per-centroid counts;
        # optimize_ivf (indexing/utils.py:24-48): map to pids and keep the sorted unique pids per centroid.
        # Both collapse to: the sorted unique (centroid, pid) pairs.
        emb2pid = torch.repeat_interleave(torch.arange(n_p, dtype=torch.int64), doclens)
        uniq = torch.unique(codes.to(dev).long() * (n_p + 1) + emb2pid.to(dev)).cpu()
        ivf = (uniq % (n_p + 1)).to(torch.int32)
        ivf_lengths = torch.bincount(uniq // (n_p + 1), minlength=K)
        return cls(centroids.cpu(), bucket_cutoffs.cpu(), bucket_weights.cpu(), codes, residuals, doclens, ivf,
                   ivf_lengths, nbits, embs.size(1))

    # -- the reference's on-disk format -----------------------------------------------------------
    @classmethod
    def load(cls, index_path):
        """Read a reference-format index directory (SURVEY.md Appendix C; index_loader.py:20-78)."""
        meta = json.load(open(os.path.join(index_path, "metadata.json")))
        nbits, dim = int(meta["config"]["nbits"]), int(meta["config"].get("dim", 128))
        centroids = torch.load(os.path.join(index_path, "centroids.pt"), map_location="cpu")
        cutoffs, weights = torch.load(os.path.join(index_path, "buckets.pt"), map_location="cpu")
        codes, residuals, doclens = [], [], []
        for c in range(int(meta["num_chunks"])):
            codes.append(torch.load(os.path.join(index_path, "%d.codes.pt" % c), map_location="cpu"))
            residuals.append(torch.load(os.path.join(index_path, "%d.residuals.pt" % c), map_location="cpu"))
            doclens.extend(json.load(open(os.path.join(index_path, "doclens.%d.json" % c))))
        ivf, ivf_lengths = torch.load(os.path.join(index_path, "ivf.pid.pt"), map_location="cpu")
        return cls(centroids, cutoffs, weights, torch.cat(codes), torch.cat(residuals), doclens, ivf, ivf_lengths,
                   nbits, dim)

    def to_npz(self):
        return dict(centroids=self.centroids.numpy(), bucket_cutoffs=self.bucket_cutoffs.numpy(),
                    bucket_weights=self.bucket_weights.numpy(), codes=self.codes.numpy(),
                    residuals=self.residuals.numpy(), doclens=self.doclens.numpy(), ivf=self.ivf.numpy(),
                    ivf_lengths=self.ivf_lengths.numpy(), nbits=np.int64(self.nbits))

    @classmethod
    def from_npz(cls, z, prefix=""):
        t = lambda k: torch.from_numpy(np.ascontiguousarray(z[prefix + k]))
        return cls(t("centroids"), t("bucket_cutoffs"), t("bucket_weights"), t("codes"), t("residuals"),
                   t("doclens"), t("ivf"), t("ivf_lengths"), int(z[prefix + "nbits"]))

    def decompress_all(self):
        """Every embedding of the index, decoded and L2-normalised (what exhaustive scoring sees)."""
        pids = torch.arange(self.doclens.numel(), dtype=torch.int32)
        return decompress(self, pids)


# ----------------------------------------------------------------------------------------------
# search
# ----------------------------------------------------------------------------------------------
def decompress(index: PlaidIndex, pids: torch.Tensor, compiled: bool | None = None) -> torch.Tensor:
    """index_storage.py:160-173: decompress_residuals_cpp over `pids` (int32), then fp32 L2 normalise.

    `compiled`: use the reference's compiled kernel (True) or decompress_residuals_restated (False);
    None = the compiled kernel when oracle/_ref holds it."""
    if compiled is None:
        compiled = have_reference_kernels()
    if compiled:
        D = _ext("decompress_residuals_cpp").decompress_residuals_cpp(
            pids, index.doclens, index.offsets, index.bucket_weights, index.reversed_bit_map, index.lut,
            index.residuals, index.codes, index.centroids, index.dim, index.nbits)
    else:
        D = decompress_residuals_restated(index, pids)
    return torch.nn.functional.normalize(D.to(torch.float32), p=2, dim=-1)


def _token_rows(index: PlaidIndex, pids: torch.Tensor) -> torch.Tensor:
    """Embedding ids of the passages `pids`, passage by passage, in token order."""
    pids = pids.long()
    lengths = index.doclens[pids]
    starts = torch.repeat_interleave(index.offsets[pids], lengths)
    first = torch.repeat_interleave(torch.cumsum(lengths, 0) - lengths, lengths)
    return starts + torch.arange(int(lengths.sum())) - first


def decompress_residuals_restated(index: PlaidIndex, pids: torch.Tensor) -> torch.Tensor:
    """torch restatement of search/decompress_residuals.cpp: for every token of every passage in `pids`,
    each residual byte goes through reversed_bit_map, then the lookup table gives its 8/nbits bucket
    indices; output[t, d] = bucket_weights[bucket index of d] + centroids[code of t, d] (fp32, unnormalised)."""
    rows = _token_rows(index, pids)
    buckets = index.lut[index.reversed_bit_map[index.residuals[rows].long()].long()].reshape(rows.numel(), index.dim)
    return index.bucket_weights[buckets.long()] + index.centroids[index.codes[rows].long()]


def segmented_lookup_restated(ivf, cells, lengths, offsets) -> torch.Tensor:
    """torch restatement of search/segmented_lookup.cpp: ivf[offsets[i] : offsets[i] + lengths[i]] of every
    cell, concatenated in cell order."""
    return torch.cat([ivf[int(o): int(o) + int(n)] for o, n in zip(offsets.tolist(), lengths.tolist())]
                     + [ivf[:0]])


def filter_pids_np(pids, centroid_scores, codes, doclens, offsets, idx, ndocs):
    """numpy restatement of search/filter_pids.cpp:27-170 (the centroid-only pruning of PLAID).

    Stage 1 (:139-141): approximate score of a passage = sum over query vectors of the max, over the
    passage's DISTINCT codes c with idx[c] set, of centroid_scores[c, k]; each per-vector max starts at
    -9999 (:30-33), so a passage with no surviving code scores -9999 * nq.  Keep the `ndocs` best by
    (score, pid) descending — std::priority_queue<pair<float,int>> order (:112-128).
    Stage 2 (:143-153): re-score those with every centroid allowed, keep ndocs // 4, same order.
    Undefined in the reference when fewer than `ndocs` candidates exist (top() of an empty queue,
    SURVEY.md hazard 2); this restatement raises instead."""
    pids = np.asarray(pids, dtype=np.int64)
    cs = np.asarray(centroid_scores, dtype=np.float32)
    codes, doclens, offsets = np.asarray(codes), np.asarray(doclens), np.asarray(offsets)

    def stage(cands, allowed, keep):
        if len(cands) < keep:
            raise ValueError("filter_pids: %d candidates < %d requested (undefined in the reference)" % (len(cands), keep))
        scored = []
        for pid in cands:
            c = np.unique(codes[offsets[pid]: offsets[pid] + doclens[pid]])
            c = c[allowed[c]]
            per_vec = np.full(cs.shape[1], -9999.0, dtype=np.float32)
            if len(c):
                per_vec = np.maximum(per_vec, cs[c].max(axis=0))
            scored.append((np.cumsum(per_vec, dtype=np.float32)[-1], int(pid)))   # sequential fp32 sum (:58-62)
        scored.sort(reverse=True)
        return [p for _, p in scored[:keep]]

    first = stage(pids, np.asarray(idx, dtype=bool), ndocs)
    return np.asarray(stage(first, np.ones(cs.shape[0], dtype=bool), ndocs // 4), dtype=np.int32)


class PlaidSearcher:
    """IndexScorer (CPU, `use_gpu=False`) over a PlaidIndex, built on the reference's compiled kernels, or on
    their restatements in this module where oracle/_ref does not hold them (`compiled` says which)."""

    def __init__(self, index: PlaidIndex, compiled: bool | None = None):
        self.index = index
        self.compiled = have_reference_kernels() if compiled is None else bool(compiled)

    def get_cells(self, Q, ncells):
        """candidate_generation.py:11-20.  Q [nq,128] fp32 -> (unique cell ids, centroid scores [K,nq])."""
        scores = self.index.centroids @ Q.T
        if ncells == 1:
            cells = scores.argmax(dim=0, keepdim=True).permute(1, 0)
        else:
            cells = scores.topk(ncells, dim=0, sorted=False).indices.permute(1, 0)
        return cells.flatten().contiguous().unique(sorted=False), scores

    def retrieve(self, Q, ncells, query_maxlen):
        """index_storage.py:66-80 + candidate_generation.py:30-36, 45-62: sorted unique candidate pids.

        Only the first `query_maxlen` query vectors select cells (:77); the IVF lookup is the reference's
        segmented_lookup_cpp over (lengths[cells], offsets[cells]) (strided_tensor.py:60-97, CPU branch)."""
        ix = self.index
        Qc = Q[:, :query_maxlen].squeeze(0)
        assert Qc.dim() == 2
        cells, centroid_scores = self.get_cells(Qc, ncells)
        cells = cells.long()
        lookup = (_ext("segmented_lookup_cpp").segmented_lookup_cpp if self.compiled
                  else segmented_lookup_restated)
        pids = lookup(ix.ivf, cells, ix.ivf_lengths[cells], ix.ivf_offsets[cells])
        pids = torch.unique_consecutive(pids.sort().values)
        return pids, centroid_scores

    def score_pids(self, Q, pids, centroid_scores, threshold, ndocs):
        """index_storage.py:102-182, CPU branch, Q.size(0) == 1."""
        ix = self.index
        idx = centroid_scores.max(-1).values >= threshold                                        # :114
        if self.compiled:
            pids = _ext("filter_pids_cpp").filter_pids_cpp(pids, centroid_scores, ix.codes, ix.doclens,
                                                           ix.offsets, idx, ndocs)              # :153-156
        else:
            pids = torch.from_numpy(filter_pids_np(pids.numpy(), centroid_scores.numpy(), ix.codes.numpy(),
                                                   ix.doclens.numpy(), ix.offsets.numpy(), idx.numpy(), ndocs))
        D_packed = decompress(ix, pids, self.compiled)                                           # :160-173
        D_lengths = ix.doclens[pids.long()]                                                      # :174
        scores = D_packed @ Q.squeeze(0).to(dtype=D_packed.dtype).T                              # colbert.py:303-305
        if self.compiled:
            return _ext("segmented_maxsim_cpp").segmented_maxsim_cpp(scores, D_lengths), pids   # colbert.py:311
        return torch.from_numpy(maxsim_oracle.segmented_maxsim(scores.numpy(), D_lengths.numpy())), pids

    def rank(self, Q, ncells=2, threshold=0.45, ndocs=1024, query_maxlen=32):
        """IndexScorer.rank (index_storage.py:86-100) for one query Q [1,Nq,128] fp32 -> (pids, scores) lists.

        Defaults are Searcher.dense_search's for k <= 10 (colbert/searcher.py:112-119)."""
        assert Q.dim() == 3 and Q.size(0) == 1
        with torch.inference_mode():
            pids, centroid_scores = self.retrieve(Q, ncells, query_maxlen)
            scores, pids = self.score_pids(Q, pids, centroid_scores, threshold, ndocs)
            order = scores.sort(descending=True)
            return pids[order.indices].tolist(), order.values.tolist()
