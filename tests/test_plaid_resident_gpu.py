"""GPU: PLAID indexes searched while they stay compressed in HBM (flmr_corpus_create_plaid + the decoding scan
kernel).  Every result is held against the decoded path of the SAME index — decode into bf16 with
flmr_plaid_decode, then the bf16 scan — and must be bit-identical: scores, top-k scores and ids, rankings,
gathered embeddings."""
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN_DIR
from oracle import maxsim_oracle as O

pytestmark = pytest.mark.gpu

CALLSITE_INDEX = os.path.join(GOLDEN_DIR, "callsites", "ckpt", "temp_index_0", "indexes", "temp_index.nbits=8")
INDEXES = [os.path.join(GOLDEN_DIR, "plaid_nbits%d" % n) for n in (1, 2, 4, 8)] + [CALLSITE_INDEX]


def _load(path, mode, **kw):
    import ravqa_b200 as R
    from ravqa_b200 import plaid
    plaid.debug_set_residency(mode)
    try:
        return R.FlatCorpus.from_plaid(path, device=0, **kw)
    finally:
        plaid.debug_set_residency("auto")


def _queries(B, nq, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    Q = torch.randn(B, nq, 128, device="cuda", generator=g)
    return torch.nn.functional.normalize(Q, dim=-1).to(torch.bfloat16)


@pytest.mark.parametrize("path", INDEXES, ids=lambda p: os.path.basename(p))
def test_compressed_index_scores_and_topk_equal_decoded(path):
    import ravqa_b200 as R
    dec, cmp = _load(path, "decoded"), _load(path, "compressed")
    try:
        assert not dec.compressed and cmp.compressed and cmp.info.hbm_bytes < dec.info.hbm_bytes
        n = cmp.n_passages
        for nq, B, seed in [(32, 3, 1), (320, 2, 2)]:
            Q = _queries(B, nq, seed)
            for relu in (False, True):
                np.testing.assert_array_equal(R.maxsim_scores(cmp, Q, relu=relu).cpu().numpy(),
                                              R.maxsim_scores(dec, Q, relu=relu).cpu().numpy())
            for k in (1, 5, 128, n + 3):
                if k <= 128:
                    cs, cp = R.maxsim_topk(cmp, Q, k)
                    ds, dp = R.maxsim_topk(dec, Q, k)
                else:      # above the fused capacity: dense scores + flmr_topk_select
                    cs, cp = R.topk_select(R.maxsim_scores(cmp, Q), k, cmp.pid_base)
                    ds, dp = R.topk_select(R.maxsim_scores(dec, Q), k, dec.pid_base)
                np.testing.assert_array_equal(cs.cpu().numpy(), ds.cpu().numpy())
                np.testing.assert_array_equal(cp.cpu().numpy(), dp.cpu().numpy())
        Q = _queries(2, 32, 9)
        cs, cp = R.topk_select(R.maxsim_scores(cmp, Q), 200)
        ds, dp = R.topk_select(R.maxsim_scores(dec, Q), 200)
        assert torch.equal(cs, ds) and torch.equal(cp, dp)
    finally:
        dec.close()
        cmp.close()


def test_executor_search_lines_give_the_same_ranking_compressed():
    """The FLMR_executor.py:774-792 search lines (as tests/test_callsites_gpu.py runs them) on the call-site index,
    once decoded and once kept compressed: the same Ranking."""
    from ravqa_b200 import ColBERTConfig, Queries, Run, RunConfig, Searcher, plaid
    z = np.load(os.path.join(GOLDEN_DIR, "callsites.npz"))
    query_embeddings = torch.from_numpy(z["queries"])
    question_ids = ["q%d" % i for i in range(query_embeddings.shape[0])]
    k = int(z["k"])
    out = {}
    for mode in ("decoded", "compressed"):
        plaid.debug_set_residency(mode)
        try:
            with Run().context(RunConfig(nranks=1, rank=0, root=os.path.join(GOLDEN_DIR, "callsites", "ckpt"),
                                         experiment="temp_index_0")):
                config = ColBERTConfig(total_visible_gpus=1)
                searcher = Searcher(index="temp_index.nbits=8", config=config)
                assert searcher.corpus.compressed == (mode == "compressed")
                queries = Queries(data={q: "question %s" % q for q in question_ids})
                ranking = searcher._search_all_Q(queries, query_embeddings, k=k)
                out[mode] = ranking.todict()
                del searcher
        finally:
            plaid.debug_set_residency("auto")
    assert out["decoded"] == out["compressed"]


def _synthetic(n_passages, nbits, seed, K=4096, lo=1, hi=96):
    """Seeded, device-generated PLAID-format shard with ragged doclens (most not multiples of 4)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    doclens = np.random.default_rng(seed).integers(lo, hi + 1, size=n_passages).astype(np.int32)
    n_tok = int(doclens.sum())
    centroids = torch.nn.functional.normalize(torch.randn(K, 128, device="cuda", generator=g), dim=-1).half().float()
    weights = (torch.sort(torch.randn(1 << nbits, device="cuda", generator=g)).values * 0.05).contiguous()
    codes = torch.randint(0, K, (n_tok,), device="cuda", generator=g, dtype=torch.int32)
    residuals = torch.randint(0, 256, (n_tok, 16 * nbits), device="cuda", generator=g, dtype=torch.int32).to(torch.uint8)
    return codes, residuals, centroids, weights, doclens


def _both(codes, residuals, centroids, weights, nbits, doclens, pid_base=0):
    import ravqa_b200 as R
    from ravqa_b200.plaid import decode_chunk
    dev = torch.device("cuda", 0)
    tokens = torch.empty((codes.numel(), 128), dtype=torch.bfloat16, device=dev)
    decode_chunk(codes, residuals, centroids, weights, nbits, tokens)
    dec = R.FlatCorpus(tokens, doclens, device=dev, pid_base=pid_base)
    # packed in chunks of 997 passages: the chunked builder must give the same corpus as one append
    cmp = R.FlatCorpus.from_plaid_arrays(codes, residuals, centroids, weights, nbits, doclens, dev, pid_base,
                                         chunk_passages=997)
    assert cmp.compressed and cmp.nbits == nbits
    return dec, cmp


@pytest.mark.parametrize("nbits", [2, 8])
def test_ragged_synthetic_corpus_bit_identical(nbits):
    import ravqa_b200 as R
    codes, residuals, centroids, weights, doclens = _synthetic(120_000, nbits, seed=nbits)
    assert (doclens % 4 != 0).mean() > 0.5
    dec, cmp = _both(codes, residuals, centroids, weights, nbits, doclens)
    del codes, residuals
    try:
        for nq in (32, 320, 832):
            for B in (1, 2, 16):
                Q = _queries(B, nq, seed=nq * 100 + B)
                cs, cp = R.maxsim_topk(cmp, Q, 10)
                ds, dp = R.maxsim_topk(dec, Q, 10)
                assert torch.equal(cs, ds) and torch.equal(cp, dp), (nq, B)
                if B == 2:
                    assert torch.equal(R.maxsim_scores(cmp, Q), R.maxsim_scores(dec, Q)), (nq, B)
    finally:
        dec.close()
        cmp.close()


def test_gather_and_rescore_equal_decoded():
    import ravqa_b200 as R
    codes, residuals, centroids, weights, doclens = _synthetic(3000, 2, seed=5)
    dec, cmp = _both(codes, residuals, centroids, weights, 2, doclens, pid_base=1000)
    try:
        pids = torch.tensor([[1000, 1005, 3999], [-1, 2500, 1000 + 2999]], device="cuda")
        dt, dm = dec.gather_padded(pids)
        ct, cm = cmp.gather_padded(pids)
        assert torch.equal(dt, ct) and torch.equal(dm, cm)
        Q = _queries(3, 32, seed=11)
        out = {}
        for name, corpus in (("dec", dec), ("cmp", cmp)):
            s = R.Searcher(index=corpus)
            out[name] = s.retrieve_and_rescore(Q, n_docs=5)
        assert np.array_equal(out["dec"]["retrieved_doc_ids"], out["cmp"]["retrieved_doc_ids"])
        assert torch.equal(out["dec"]["doc_scores"], out["cmp"]["doc_scores"])
        assert torch.equal(out["dec"]["search_scores"], out["cmp"]["search_scores"])
    finally:
        dec.close()
        cmp.close()


def test_two_compressed_shards_merge_to_the_unsharded_result():
    import ravqa_b200 as R
    full = _load(CALLSITE_INDEX, "compressed")
    shards = [_load(CALLSITE_INDEX, "compressed", rank=r, world_size=2) for r in (0, 1)]
    try:
        assert all(s.compressed for s in shards) and shards[1].pid_base == shards[0].n_passages
        Q = _queries(4, 32, seed=21)
        for k in (1, 5, 50):
            parts = [R.maxsim_topk(s, Q, k) for s in shards]
            ms, mp = R.topk_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]), k)
            fs, fp = R.maxsim_topk(full, Q, k)
            assert torch.equal(ms, fs) and torch.equal(mp, fp), k
    finally:
        full.close()
        for s in shards:
            s.close()


def test_search_on_compressed_corpus_is_cuda_graph_capturable():
    import ravqa_b200 as R
    cmp = _load(os.path.join(GOLDEN_DIR, "plaid_nbits2"), "compressed")
    try:
        Qs = _queries(3, 320, seed=1)
        R.maxsim_topk(cmp, Qs, 5)
        R.maxsim_scores(cmp, Qs)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            gs, gp = R.maxsim_topk(cmp, Qs, 5)
            ga = R.maxsim_scores(cmp, Qs)
        for seed in (2, 3):
            Qs.copy_(_queries(3, 320, seed=seed))
            graph.replay()
            torch.cuda.synchronize()
            es, ep = R.maxsim_topk(cmp, Qs, 5)
            assert torch.equal(gs, es) and torch.equal(gp, ep) and torch.equal(ga, R.maxsim_scores(cmp, Qs))
    finally:
        cmp.close()


def test_corrupt_code_is_rejected_at_creation():
    from ravqa_b200 import _cabi
    from ravqa_b200.plaid import create_compressed
    codes, residuals, centroids, weights, doclens = _synthetic(50, 4, seed=3, K=64)
    codes[7] = 64                                              # one past the last centroid
    with pytest.raises(_cabi.FlmrError, match="centroid code"):
        create_compressed(codes, residuals, centroids, weights, 4, doclens, torch.device("cuda", 0))
    codes[7] = -1
    with pytest.raises(_cabi.FlmrError, match="centroid code"):
        create_compressed(codes, residuals, centroids, weights, 4, doclens, torch.device("cuda", 0))


def test_simt_cross_check_reports_unsupported_for_compressed():
    import ravqa_b200 as R
    from ravqa_b200 import _cabi
    cmp = _load(os.path.join(GOLDEN_DIR, "plaid_nbits8"), "compressed")
    try:
        with pytest.raises(_cabi.FlmrError) as e:
            R.debug_scores_simt(cmp, _queries(1, 32, seed=1))
        assert e.value.code == 3
    finally:
        cmp.close()


def test_compressed_corpus_matches_the_oracle_on_the_fixture():
    """Anchor: the compressed path also agrees with the fp32 oracle over the reference's decoded embeddings."""
    import ravqa_b200 as R
    z = np.load(os.path.join(GOLDEN_DIR, "plaid_nbits8.npz"))
    cmp = _load(os.path.join(GOLDEN_DIR, "plaid_nbits8"), "compressed")
    try:
        Q, _, _ = O.synth(1, 4, 3, 32, seed=3)
        ref = O.maxsim_scores(Q, O.bf16_round(z["decoded_ref"]), z["doclens"])
        got = R.maxsim_scores(cmp, torch.from_numpy(Q)).cpu().numpy()
        np.testing.assert_allclose(got, ref, rtol=2e-4, atol=1e-4)
    finally:
        cmp.close()


def _write_plaid_dir(path, n_chunks, passages_per_chunk, nbits, seed, K=1024):
    """A PLAID index directory in the reference's layout with several chunks (seeded, generated on the GPU)."""
    import json
    g = torch.Generator(device="cuda").manual_seed(seed)
    rng = np.random.default_rng(seed)
    os.makedirs(path, exist_ok=True)
    cent = torch.nn.functional.normalize(torch.randn(K, 128, device="cuda", generator=g), dim=-1).half()
    torch.save(cent.cpu(), os.path.join(path, "centroids.pt"))
    weights = torch.sort(torch.randn(1 << nbits, device="cuda", generator=g)).values * 0.05
    torch.save((torch.zeros((1 << nbits) - 1), weights.half().cpu()), os.path.join(path, "buckets.pt"))
    n_emb = 0
    for c in range(n_chunks):
        dl = rng.integers(1, 120, size=passages_per_chunk)
        n = int(dl.sum())
        n_emb += n
        torch.save(torch.randint(0, K, (n,), device="cuda", generator=g, dtype=torch.int32).cpu(),
                   os.path.join(path, "%d.codes.pt" % c))
        torch.save(torch.randint(0, 256, (n, 16 * nbits), device="cuda", generator=g,
                                 dtype=torch.int32).to(torch.uint8).cpu(), os.path.join(path, "%d.residuals.pt" % c))
        with open(os.path.join(path, "doclens.%d.json" % c), "w") as f:
            json.dump([int(x) for x in dl], f)
    with open(os.path.join(path, "metadata.json"), "w") as f:
        json.dump({"config": {"nbits": nbits, "dim": 128}, "num_chunks": n_chunks, "num_embeddings": n_emb}, f)
    return n_emb


def test_compressed_load_peak_memory_is_resident_plus_one_chunk(tmp_path):
    """from_plaid on a multi-chunk index stages ONE chunk at a time: torch's peak during the load stays within
    one chunk's codes + residuals (+ centroids and their fp32 upcast), and nothing stays cached afterwards; the
    loaded corpus searches exactly like the decoded one."""
    import ravqa_b200 as R
    nbits, n_chunks, per = 4, 6, 4000
    path = str(tmp_path / "idx")
    n_emb = _write_plaid_dir(path, n_chunks, per, nbits, seed=7)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    cmp = _load(path, "compressed")
    try:
        peak = torch.cuda.max_memory_allocated() - base
        chunk_bytes = (n_emb / n_chunks) * (4 + 16 * nbits)
        centroid_bytes = 1024 * 128 * (2 + 4)
        assert peak <= 1.5 * chunk_bytes + centroid_bytes + (1 << 20), (peak, chunk_bytes)
        assert peak < 0.5 * n_emb * (4 + 16 * nbits)          # not the whole shard
        assert torch.cuda.memory_reserved() - torch.cuda.memory_allocated() < (8 << 20)   # staging released
        rows = int(cmp.info.n_rows) + 96
        assert cmp.info.hbm_bytes >= rows * (8 + 16 * nbits)
        dec = _load(path, "decoded")
        try:
            Q = _queries(4, 64, seed=3)
            cs, cp = R.maxsim_topk(cmp, Q, 20)
            ds, dp = R.maxsim_topk(dec, Q, 20)
            assert torch.equal(cs, ds) and torch.equal(cp, dp)
        finally:
            dec.close()
        # a shard of it: only its chunks' passages
        sh = _load(path, "compressed", rank=1, world_size=3)
        try:
            assert sh.compressed and sh.pid_base > 0
        finally:
            sh.close()
    finally:
        cmp.close()


def test_builder_append_must_hold_whole_passages():
    from ravqa_b200 import _cabi
    from ravqa_b200.plaid import _append, _builder_from
    codes, residuals, centroids, weights, doclens = _synthetic(40, 2, seed=4, K=64)
    dev = torch.device("cuda", 0)
    L = _cabi.lib()
    b = _builder_from(centroids, weights, 2, doclens, dev, 0)
    try:
        with pytest.raises(_cabi.FlmrError, match="whole passages"):
            _append(b, codes[:int(doclens[0]) + 1], residuals[:int(doclens[0]) + 1])
        _append(b, codes[:int(doclens[0])], residuals[:int(doclens[0])])
        import ctypes as C
        h = C.c_void_p()
        assert L.flmr_corpus_plaid_builder_finish(b, C.byref(h)) == 1      # 39 passages still missing
        assert "of 40 passages" in L.flmr_last_error().decode()
    finally:
        L.flmr_corpus_plaid_builder_destroy(b)
