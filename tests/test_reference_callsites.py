"""CPU: the reference's call sites and methods driven through this repository's host layer — index addressing,
PLAID auto-detection, the literal call sites of src/executors/FLMR_executor.py:774-792 and
src/models/rag/rag_model_blip.py:297-301, 397, 430-435, ``ColBERT.score`` / ``ColBERT.compute_ib_loss_new`` after
``integration.patch_colbert()`` — against what the reference's own code returned for the same inputs.

The reference package is not needed: the ``colbert`` modules these lines import are stand-ins holding this package's
duck-typed ``Run`` / ``RunConfig`` / ``ColBERTConfig`` / ``Queries`` (``ravqa_b200.infra``) and placeholders for the
objects ``patch_colbert()`` replaces, and the reference's results (index paths, scores, gradients) are goldens
recorded from the reference by tests/golden/make_golden_reference_checks.py and make_golden_callsites.py.

There is no GPU here, so the lowest layer (the C-ABI calls of maxsim.py / corpus.py) is substituted by the
numpy oracle — test infrastructure, tests/oracle_backend.py.  The same lines run on the GPU box against the real
kernels in tests/test_callsites_gpu.py.
"""
import contextlib
import json
import os
import random
import sys
import types

import numpy as np
import pytest
import torch

from helpers import GOLDEN_DIR

sys.path.insert(0, GOLDEN_DIR)
import make_golden_reference_checks as G  # noqa: E402

CKPT_DIR = os.path.join(GOLDEN_DIR, "callsites", "ckpt")


@pytest.fixture()
def ref(monkeypatch):
    """Stand-ins for the ``colbert`` modules the call sites import (installed for one test)."""
    import ravqa_b200.infra as I
    # the oracle backend computes on the host, so the host layer must take its CPU route on a GPU machine too
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)

    def module(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        monkeypatch.setitem(sys.modules, name, m)
        return m

    class Searcher:                 # placeholders: patch_colbert() rebinds them, nothing calls them
        pass

    class Indexer:
        pass

    class Checkpoint:
        pass

    def colbert_score(Q, D_padded, D_mask, config=None):
        raise AssertionError("the reference's colbert_score is not available here: patch_colbert() first")

    def colbert_score_packed(Q, D_packed, D_lengths, config=None):
        raise AssertionError("the reference's colbert_score_packed is not available here: patch_colbert() first")

    def compute_ib_loss_new(self, Q, D, D_mask):
        raise AssertionError("the reference's compute_ib_loss_new is not available here: patch_colbert() first")

    M = module("colbert.modeling.colbert", colbert_score=colbert_score, colbert_score_packed=colbert_score_packed)

    class ColBERT:
        def score(self, Q, D_padded, D_mask):
            # colbert.py:217-224 (cosine similarity): the module-level colbert_score with the model's config
            return M.colbert_score(Q, D_padded, D_mask, config=self.colbert_config)

    ColBERT.compute_ib_loss_new = compute_ib_loss_new
    M.ColBERT = ColBERT
    infra = module("colbert.infra", Run=I.Run, RunConfig=I.RunConfig, ColBERTConfig=I.ColBERTConfig)
    data = module("colbert.data", Queries=I.Queries)
    S = module("colbert.searcher", Searcher=Searcher)
    IX = module("colbert.indexer", Indexer=Indexer)
    CK = module("colbert.modeling.checkpoint", Checkpoint=Checkpoint)
    modeling = module("colbert.modeling", colbert=M, checkpoint=CK)
    return module("colbert", Searcher=Searcher, Indexer=Indexer, infra=infra, data=data, searcher=S, indexer=IX,
                  modeling=modeling)


@pytest.fixture()
def golden():
    z = np.load(os.path.join(GOLDEN_DIR, "callsites.npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def recorded():
    """What the reference's own code returned (tests/golden/make_golden_reference_checks.py)."""
    z = np.load(os.path.join(GOLDEN_DIR, "reference_checks.npz"))
    return {k: z[k] for k in z.files}


# ---------------------------------------------------------------------------------------------------------
# index addressing
# ---------------------------------------------------------------------------------------------------------
def test_index_path_resolution_equals_reference(recorded):
    """infra.resolve_index_path == os.path.join(ColBERTConfig.from_existing(config, Run().config).index_root_, index)
    (colbert/searcher.py:26-30) as the reference computed it for its own config / Run objects: the duck-typed infra
    classes give the same answers in the same situations."""
    import ravqa_b200.infra as I
    cwd = os.path.dirname(I._RUN_FIELDS["root"])     # (without a context: <cwd at import>/experiments/default/indexes/)
    scenarios = json.loads(str(recorded["paths_json"]))
    assert [[s["stack"], s["config"]] for s in scenarios] == json.loads(json.dumps(G.PATH_SCENARIOS))
    for sc in scenarios:
        stack, ckw = sc["stack"], sc["config"]
        with contextlib.ExitStack() as es:
            for kw in stack:
                es.enter_context(I.Run().context(I.RunConfig(**kw)))
            own = I.resolve_index_path("temp_index.nbits=8", I.ColBERTConfig(**ckw))
            want = sc["want"].replace("<cwd>", cwd, 1)
            assert os.path.normpath(own) == os.path.normpath(want), (stack, ckw, own, want)
            # absolute index names win over any root, as os.path.join makes them do in the reference
            assert I.resolve_index_path("/abs/idx", I.ColBERTConfig(**ckw)) == sc["want_abs"] == "/abs/idx"
    # from_existing / assigned semantics of the stand-ins (core_config.py:20-36, base_config.py:20-35)
    a = I.ColBERTConfig(nbits=8, doc_maxlen=None)
    assert set(a.assigned) == {"nbits", "doc_maxlen"} and a.doc_maxlen == 220     # None -> default, still assigned
    b = I.ColBERTConfig.from_existing(a, I.RunConfig(root="/r"))
    assert b.nbits == 8 and b.root == "/r" and "experiment" not in b.assigned
    b.configure(ncells=2, bogus=1)
    assert b.ncells == 2 and "ncells" in b.assigned and not hasattr(b, "bogus")
    assert len(I.Run().stack) == 1                                                 # contexts popped


def test_index_kind_detection(tmp_path):
    import ravqa_b200 as R
    from ravqa_b200.searcher import detect_index_kind
    plaid = os.path.join(CKPT_DIR, "temp_index_0", "indexes", "temp_index.nbits=8")
    assert detect_index_kind(plaid) == "plaid"
    flat = str(tmp_path / "flat")
    R.save_flat_index(flat, torch.zeros(6, 128, dtype=torch.bfloat16), [2, 4])
    assert detect_index_kind(flat) == "flat"
    only_plan = tmp_path / "building"
    only_plan.mkdir()
    (only_plan / "plan.json").write_text("{}")
    with pytest.raises(ValueError, match="did not finish"):
        detect_index_kind(str(only_plan))
    with pytest.raises(FileNotFoundError):
        detect_index_kind(str(tmp_path / "missing"))
    # the index config comes from where the reference reads it (base_config.py:71-87)
    cfg = R.ColBERTConfig.load_from_index(plaid)
    assert cfg.nbits == 8 and cfg.dim == 128 and cfg.index_name == "temp_index.nbits=8"


# ---------------------------------------------------------------------------------------------------------
# the literal call sites, reference objects + this repository's Searcher
# ---------------------------------------------------------------------------------------------------------
def test_executor_search_lines_verbatim_with_patched_colbert(ref, golden, monkeypatch):
    """FLMR_executor.py:774-792, copied line by line, with ``from colbert import Searcher`` resolved AFTER
    ``patch_colbert()``; Run / RunConfig / ColBERTConfig / Queries come from the ``colbert`` modules."""
    import oracle_backend
    import ravqa_b200.integration as flmr_b200
    oracle_backend.install(monkeypatch)
    import colbert.searcher
    original = colbert.searcher.Searcher
    # an executor that did `from colbert import Indexer, Searcher` BEFORE the patch (FLMR_executor.py:47)
    import types
    early = types.ModuleType("an_executor_imported_earlier")
    early.Searcher = original
    sys.modules[early.__name__] = early
    try:
        done = flmr_b200.patch_colbert()
        assert done["Searcher"] >= 3 and early.Searcher is flmr_b200.Searcher   # colbert, colbert.searcher, the executor
        from colbert import Searcher
        from colbert.data import Queries
        from colbert.infra import ColBERTConfig, Run, RunConfig
        import ravqa_b200
        assert Searcher is ravqa_b200.Searcher

        # ---- names the executor has in scope at that point ----
        class _Self:
            global_rank = 0
            device = torch.device("cpu")            # (the reference then asks for total_visible_gpus = 0)
            config = type("C", (), {"ckpt_dir": CKPT_DIR})()
            model_config = {"nbits": 8}
        self = _Self()
        dataloader_idx = 0
        question_ids = ["q%d" % i for i in range(golden["queries"].shape[0])]
        questions = ["question %d" % i for i in range(len(question_ids))]
        query_embeddings = torch.from_numpy(golden["queries"])
        Ks = [1, 5, int(golden["k"])]
        get_world_size = lambda: 1                  # noqa: E731

        # ---- FLMR_executor.py:774-792, verbatim (minus logging and the distributed barrier) ----
        with Run().context(RunConfig(nranks=1, rank=self.global_rank, root=self.config.ckpt_dir, experiment=f"temp_index_{dataloader_idx}")):
            if self.device == torch.device('cpu'):
                total_visible_gpus = 0
            else:
                if get_world_size() > 1:
                    total_visible_gpus = 0
                else:
                    total_visible_gpus = 1 #torch.cuda.device_count()

            config = ColBERTConfig(
                total_visible_gpus=total_visible_gpus,
            )
            nbits = self.model_config.get("nbits", 2)
            searcher = Searcher(index=f"temp_index.nbits={nbits}", config=config)
            custom_quries = {question_id: question for question_id, question in zip(question_ids, questions)}
            queries = Queries(data=custom_quries)
            ranking = searcher._search_all_Q(queries, query_embeddings, k=max(Ks))

            ranking_dict = ranking.todict()

            del searcher
        # ---- what the lines after it consume (FLMR_executor.py:851-878) ----
        assert list(ranking_dict.keys()) == question_ids
        want = np.argsort(-golden["exact_scores_bf16"], axis=1, kind="stable")[:, :max(Ks)]
        for qi, (question_id, ranking_list) in enumerate(zip(question_ids, ranking_dict.values())):
            assert len(ranking_list) == max(Ks)
            for rank0, entry in enumerate(ranking_list):
                retrieved_doc_index, rank, retrieved_doc_score = entry
                assert isinstance(retrieved_doc_index, int) and rank == rank0 + 1 and isinstance(retrieved_doc_score, float)
            assert [e[0] for e in ranking_list] == want[qi].tolist()
            np.testing.assert_allclose([e[2] for e in ranking_list], golden["exact_scores_bf16"][qi, want[qi]], rtol=5e-4)
        assert ranking.provenance()["source"] == "Searcher::search_all"
    finally:
        flmr_b200.unpatch_colbert()
        sys.modules.pop(early.__name__, None)
    assert colbert.searcher.Searcher is original and ref.Searcher is original


def test_rag_retrieval_lines_verbatim_with_patched_colbert(ref, golden, recorded, monkeypatch):
    """rag_model_blip.py:288-301 (index opened through the Run context derived from ``index_path``) and
    :390-441 (search, per-question re-score through ``ColBERT.score``), with the backend patched in; result =
    what the unpatched reference computed for the same retrieved passages."""
    import oracle_backend
    import ravqa_b200.integration as flmr_b200
    oracle_backend.install(monkeypatch)
    from colbert.modeling.colbert import ColBERT
    from colbert.infra import ColBERTConfig as RC
    # host dictionary of item embeddings, as rag_model_blip.py:303-330 loads it: pid -> (emb [Nd, d], mask [Nd, 1]),
    # bf16-exact, so both sides see identical operands
    item_embeddings = G.rag_item_embeddings(golden["doclens"])

    class _Encoder:          # ColBERT.score bound to a stand-in `self` (no BERT weights offline)
        colbert_config = RC(total_visible_gpus=0)
        use_gpu = False
        score = ColBERT.score

    def run_lines():
        from colbert import Searcher
        from colbert.data import Queries
        from colbert.infra import ColBERTConfig, Run, RunConfig

        class _Self:
            global_rank = 0
            device = torch.device("cpu")
            question_encoder = _Encoder()
        self = _Self()
        self.item_embeddings = item_embeddings
        index_path = os.path.join(CKPT_DIR, "temp_index_0")
        # ---- rag_model_blip.py:288-301 ----
        index_root = os.path.dirname(index_path)
        index_name = os.path.basename(index_path)
        if self.device == torch.device('cpu'):
            total_visible_gpus = 0
        else:
            total_visible_gpus = 1
        with Run().context(RunConfig(nranks=1, rank=self.global_rank, root=index_root, experiment=index_name)):
            config = ColBERTConfig(
                total_visible_gpus=total_visible_gpus,
            )
            self.index = Searcher(index=f"temp_index.nbits=8", config=config)
        # ---- rag_model_blip.py:388-441 ----
        question_hidden_states = torch.from_numpy(golden["queries"]).clone().requires_grad_(True)
        input_text_sequences = ["question %d" % i for i in range(question_hidden_states.size(0))]
        n_docs = 3
        custom_quries = {i: query for i, query in enumerate(input_text_sequences)}
        queries = Queries(data=custom_quries)
        if n_docs < 5:
            n_docs_retrieve = 5
        else:
            n_docs_retrieve = n_docs
        ranking = self.index._search_all_Q(queries, question_hidden_states.cpu().detach(), k=n_docs_retrieve, progress=False)
        retrieval_results = ranking.todict()
        doc_scores = []
        all_retrieved_doc_indices = []
        for query_index, retrieved_docs in retrieval_results.items():
            retrieved_doc_indices = []
            retrieved_doc_scores = []
            if n_docs != n_docs_retrieve:
                retrieved_docs = random.sample(retrieved_docs, n_docs)
            for doc_index, _, doc_score in retrieved_docs:
                retrieved_doc_indices.append(doc_index)
                retrieved_doc_scores.append(doc_score)
            retrieved_item_embeddings = []
            retrieved_item_embeding_mask = []
            for i in retrieved_doc_indices:
                emb_tuple = self.item_embeddings[i]
                retrieved_item_embeddings.append(torch.Tensor(emb_tuple[0]))
                retrieved_item_embeding_mask.append(torch.Tensor(emb_tuple[1]))
            retrieved_item_embeddings = torch.stack(retrieved_item_embeddings).to(self.device)
            retrieved_item_embeding_mask = torch.stack(retrieved_item_embeding_mask).to(self.device)
            retrieved_query_embedding = question_hidden_states[[query_index]]
            self.question_encoder.colbert_config.nway = len(retrieved_doc_indices)
            Q_duplicated = retrieved_query_embedding.repeat_interleave(self.question_encoder.colbert_config.nway, dim=0).contiguous()
            scores = self.question_encoder.score(Q_duplicated, retrieved_item_embeddings, retrieved_item_embeding_mask)
            doc_scores.append(scores)
            all_retrieved_doc_indices.append(retrieved_doc_indices)
        doc_scores = torch.stack(doc_scores)
        ids = np.array(all_retrieved_doc_indices)
        doc_scores.sum().backward()
        return ids, doc_scores.detach(), question_hidden_states.grad.clone()

    try:
        flmr_b200.patch_colbert()
        random.seed(11)
        ids, doc_scores, dq = run_lines()
    finally:
        flmr_b200.unpatch_colbert()
    # retrieved ids: subsets of the exact top-5 over the reference's decompressed index, the same draw as recorded
    top5 = np.argsort(-golden["exact_scores_bf16"], axis=1, kind="stable")[:, :5]
    assert ids.shape == (golden["queries"].shape[0], 3)
    for b in range(ids.shape[0]):
        assert set(ids[b]).issubset(set(top5[b]))
    assert np.array_equal(ids, recorded["rag_ids"])
    # the re-score and its gradient: the UNPATCHED reference ColBERT.score on the same passages (fp32 autograd)
    np.testing.assert_allclose(doc_scores.numpy(), recorded["rag_scores"], rtol=1e-5)
    np.testing.assert_allclose(dq.numpy(), recorded["rag_dQ"], rtol=1e-5, atol=1e-6)


def test_reference_colbert_methods_route_into_this_backend(ref, recorded, monkeypatch):
    """``ColBERT.score`` (colbert.py:217-224) in its three caller shapes and ``ColBERT.compute_ib_loss_new``
    (colbert.py:82-113) after ``patch_colbert()``: the values and gradients the reference's own methods gave before
    the patch, and every score comes out of this repository's entry points."""
    import oracle_backend
    import ravqa_b200.integration as flmr_b200
    calls = oracle_backend.install(monkeypatch)
    from colbert.infra import ColBERTConfig as RC
    from colbert.modeling.colbert import ColBERT

    class _Model:
        colbert_config = RC(total_visible_gpus=0, nway=2, use_ib_negatives=True)
        use_gpu = False
        loss_fn = torch.nn.CrossEntropyLoss()
        score = ColBERT.score
        compute_ib_loss_new = ColBERT.compute_ib_loss_new

    try:
        flmr_b200.patch_colbert()

        class _Patched(_Model):
            score = ColBERT.score
            compute_ib_loss_new = ColBERT.compute_ib_loss_new      # now the replacement method
        after = G.methods_run(_Patched(), *G.methods_inputs())
    finally:
        flmr_b200.unpatch_colbert()
    assert calls["argmax_grouped"] >= 2 and calls["argmax"] >= 2 and calls["backward_grouped"] >= 1
    for key in ("eval", "one"):
        np.testing.assert_allclose(after[key].numpy(), recorded["methods_" + key], rtol=1e-5)
    for key in ("train_scores", "train_loss", "train_dQ", "train_dD"):
        np.testing.assert_allclose(after[key].numpy(), recorded["methods_" + key], rtol=1e-4, atol=1e-5)
    assert ColBERT.compute_ib_loss_new is _Model.__dict__["compute_ib_loss_new"]   # restored


@pytest.mark.parametrize("nq", G.FLIPR_NQ)
def test_flipr_interaction_equals_reference(ref, recorded, monkeypatch, nq):
    """``config.interaction == 'flipr'`` (colbert_score_reduce, colbert.py:248-261; unused by FLMR): this package's
    ``colbert_score`` against the reference's own — one query vs all documents and aligned pairs, values and
    gradients — with fewer than 8 (no second term), exactly 8 and more tokens beyond ``query_maxlen``."""
    import oracle_backend
    import ravqa_b200 as R
    oracle_backend.install(monkeypatch)
    from colbert.infra import ColBERTConfig as RC
    cfg = RC(total_visible_gpus=0, interaction="flipr", query_maxlen=64)
    Q0, D0, M0, w, lens = G.flipr_inputs(nq)
    for tag, q_rows in (("one", slice(0, 1)), ("all", slice(0, Q0.size(0)))):
        Q, D = Q0[q_rows].clone().requires_grad_(True), D0.clone().requires_grad_(True)
        s = R.colbert_score(Q, D, M0, config=cfg)
        (s * w).sum().backward()
        for got, key in ((s.detach(), "scores"), (Q.grad, "dQ"), (D.grad, "dD")):
            np.testing.assert_allclose(got.numpy(), recorded["flipr_%d_%s_%s" % (nq, tag, key)], rtol=1e-5, atol=1e-6)
    # and it is not the plain sum
    assert not torch.allclose(R.colbert_score(Q0[:1], D0, M0, config=cfg), R.colbert_score(Q0[:1], D0, M0))
    # packed form (colbert.py:289-311: 'flipr' always takes the padded reduction)
    import ravqa_b200.integration as I
    packed = torch.cat([D0[i, :l] for i, l in enumerate(lens)])
    got = I.colbert_score_packed(Q0[:1], packed, lens, cfg)
    np.testing.assert_allclose(got.numpy(), recorded["flipr_%d_packed" % nq], rtol=1e-5)
    with pytest.raises(NotImplementedError):
        R.Searcher(index=oracle_backend.OracleCorpus(packed, lens), config=cfg)


def test_text_search_goes_through_the_references_checkpoint(ref, golden, monkeypatch):
    """``Searcher.search`` / ``search_all`` (searcher.py:52-71) with ``checkpoint=``: the query encoder is
    ``colbert.modeling.checkpoint.Checkpoint``, constructed lazily with (name, colbert_config=
    searcher.config) and asked through ``queryFromText`` exactly as the reference's ``encode`` does — here a recording
    stand-in with the same constructor and method (no BERT weights offline) that returns the golden query
    embeddings, so the ranking is the exact one."""
    import oracle_backend
    import ravqa_b200 as R
    import colbert.modeling.checkpoint as CK
    from colbert.data import Queries
    from colbert.infra import ColBERTConfig, Run, RunConfig
    oracle_backend.install(monkeypatch)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    seen = {}
    Qg = torch.from_numpy(golden["queries"])
    texts = ["question %d" % i for i in range(Qg.size(0))]

    class FakeCheckpoint:
        def __init__(self, name, colbert_config=None):
            seen["ctor"] = (name, colbert_config)
            self.query_tokenizer = type("T", (), {"query_maxlen": None})()

        def queryFromText(self, queries, bsize=None, to_cpu=False, context=None):
            seen.setdefault("calls", []).append((list(queries), bsize, to_cpu, self.query_tokenizer.query_maxlen))
            return torch.stack([Qg[texts.index(q)] for q in queries])

    monkeypatch.setattr(CK, "Checkpoint", FakeCheckpoint)
    with Run().context(RunConfig(nranks=1, rank=0, root=CKPT_DIR, experiment="temp_index_0")):
        searcher = R.Searcher(index="temp_index.nbits=8", checkpoint="some/checkpoint",
                              config=ColBERTConfig(total_visible_gpus=0, query_maxlen=48))
    assert "ctor" not in seen                                        # nothing is loaded until text arrives
    k = int(golden["k"])
    want = np.argsort(-golden["exact_scores_bf16"], axis=1, kind="stable")[:, :k]
    pids, ranks, scores = searcher.search(texts[3], k=k)
    assert seen["ctor"][0] == "some/checkpoint" and seen["ctor"][1] is searcher.config
    assert seen["calls"][0] == ([texts[3]], None, False, 48)
    assert pids == want[3].tolist() and ranks == list(range(1, k + 1))
    ranking = searcher.search_all(Queries(data=dict(zip(["a%d" % i for i in range(len(texts))], texts))), k=k)
    assert [[e[0] for e in v] for v in ranking.todict().values()] == want.tolist()
    assert len(seen["calls"]) == 2 and seen["calls"][1][0] == texts
    # no checkpoint and no encode_fn: a clear error instead of a silent CPU path
    with Run().context(RunConfig(nranks=1, rank=0, root=CKPT_DIR, experiment="temp_index_0")):
        bare = R.Searcher(index="temp_index.nbits=8", config=ColBERTConfig(total_visible_gpus=0))
    bare.index_config.checkpoint = None
    with pytest.raises(RuntimeError, match="encode_fn"):
        bare.search("text", k=3)


def test_indexer_with_the_references_checkpoint_and_run_context(ref, monkeypatch, tmp_path):
    """``Indexer(checkpoint=..., config=...).index(name=..., collection=..., overwrite=True)`` as
    FLMR_executor.py:601-617 calls it, inside ``Run().context``: the document encoder is
    ``colbert.modeling.checkpoint.Checkpoint`` (a recording stand-in here: no BERT weights offline) driven with the batching of
    ``CollectionEncoder.encode_passages``; the flat index lands where ``config.index_path_`` points
    (``<root>/<experiment>/indexes/<name>``), and ``Searcher(index=name)`` in the same context opens and ranks it."""
    import zlib
    import oracle_backend
    import ravqa_b200 as R
    import colbert.modeling.checkpoint as CK
    from colbert.infra import ColBERTConfig, Run, RunConfig
    oracle_backend.install(monkeypatch)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    seen = {"batches": []}

    def embed(text):
        g = torch.Generator().manual_seed(zlib.crc32(text.encode()))
        n = 3 + zlib.crc32(text.encode()) % 6
        return torch.nn.functional.normalize(torch.randn(n, 128, generator=g), dim=-1)

    class FakeCheckpoint:
        def __init__(self, name, colbert_config=None):
            seen["ctor"] = (name, colbert_config)

        def docFromText(self, docs, bsize=None, keep_dims=True, to_cpu=False, showprogress=False, return_tokens=False):
            assert keep_dims == "flatten" and torch.is_inference_mode_enabled()
            seen["batches"].append((len(docs), bsize))
            embs = [embed(d) for d in docs]
            return torch.cat(embs), [e.size(0) for e in embs]

    monkeypatch.setattr(CK, "Checkpoint", FakeCheckpoint)
    collection = ["passage number %d" % i for i in range(230)]
    with Run().context(RunConfig(nranks=1, rank=0, root=str(tmp_path), experiment="temp_index_0")):
        config = ColBERTConfig(nbits=8, doc_maxlen=512, total_visible_gpus=0, bsize=2)
        indexer = R.Indexer(checkpoint="a/checkpoint", config=config)
        path = indexer.index(name="temp_index.nbits=8", collection=collection, overwrite=True)
        assert path == os.path.join(str(tmp_path), "temp_index_0", "indexes", "temp_index.nbits=8")
        assert path == ColBERTConfig.from_existing(config, Run().config).index_root_ + "temp_index.nbits=8" \
            or os.path.normpath(path) == os.path.normpath(os.path.join(
                ColBERTConfig.from_existing(config, Run().config).index_root_, "temp_index.nbits=8"))
        assert seen["ctor"] == ("a/checkpoint", config)
        assert seen["batches"] == [(100, 2), (100, 2), (30, 2)]           # bsize * 50 passages per docFromText call
        searcher = R.Searcher(index="temp_index.nbits=8", config=ColBERTConfig(total_visible_gpus=0))
    assert searcher.index_kind == "flat" and searcher.corpus.n_passages == len(collection)
    Q = torch.stack([torch.nn.functional.pad(embed(collection[i]), (0, 0, 0, 8 - embed(collection[i]).size(0)))
                     for i in (7, 100, 229)])
    ranking = searcher._search_all_Q(None, Q, k=3).todict()
    assert [v[0][0] for v in ranking.values()] == [7, 100, 229]          # each passage's own tokens find it first
    # opt-in: `from colbert import Indexer` itself becomes the flat-store Indexer; a TSV path is a collection too
    import ravqa_b200.integration as flmr_b200
    import colbert.indexer
    original = colbert.indexer.Indexer
    tsv = tmp_path / "collection.tsv"
    tsv.write_text("".join("%d\t%s\ttitle %d\n" % (i, t, i) for i, t in enumerate(collection[:20])))
    try:
        assert flmr_b200.patch_colbert(searcher=False, scoring=False, ib_loss=False, indexer=True)["Indexer"] >= 2
        from colbert import Indexer
        assert Indexer is R.Indexer
        with Run().context(RunConfig(nranks=1, root=str(tmp_path), experiment="temp_index_1")):
            indexer = Indexer(checkpoint="a/checkpoint", config=ColBERTConfig(nbits=2, bsize=4))
            indexer.index(name="temp_index.nbits=2", collection=str(tsv), overwrite=True)
            index_path = indexer.get_index()
        assert index_path == os.path.join(str(tmp_path), "temp_index_1", "indexes", "temp_index.nbits=2")
        from ravqa_b200.index_io import load_flat_index
        tokens, doclens, meta = load_flat_index(index_path)
        want = [embed("title %d | %s" % (i, t)).size(0) for i, t in enumerate(collection[:20])]
        assert doclens.tolist() == want and tokens.size(0) == sum(want)
    finally:
        flmr_b200.unpatch_colbert()
    assert colbert.indexer.Indexer is original
