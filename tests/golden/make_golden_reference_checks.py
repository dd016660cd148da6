"""Record what the reference's own code returns for the checks of tests/test_reference_callsites.py and
tests/test_oracle.py, so that those tests compare against it without the reference checkout.

    python tests/golden/make_golden_reference_checks.py <reference checkout>/third_party/ColBERT

Calls, unmodified, from third_party/ColBERT/colbert (through the import shims of make_golden.py):
    ColBERT.segmented_maxsim (segmented_maxsim.cpp)     -> segmented_*
    ColBERTConfig.from_existing(config, Run().config).index_root_ under Run().context  -> paths_json
    colbert_score / colbert_score_packed with interaction='flipr'                  -> flipr_<nq>_*
    ColBERT.score / ColBERT.compute_ib_loss_new in their three caller shapes       -> methods_*
    ColBERT.score re-scoring the passages the RAG lines retrieve                  -> rag_*
Inputs are regenerated from the same seeds by the tests (torch CPU generators, numpy for the RAG item
embeddings), so only the reference's outputs are stored.  Writes tests/golden/reference_checks.npz.
"""
from __future__ import annotations

import contextlib
import json
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))

# (RunConfig kwargs stack, ColBERTConfig kwargs) of test_index_path_resolution_equals_reference
PATH_SCENARIOS = [
    ([dict(nranks=1, rank=0, root="/ckpt", experiment="temp_index_0")], dict(total_visible_gpus=0)),
    ([dict(nranks=1, rank=3, root="/data/idx", experiment="okvqa")], dict(total_visible_gpus=1)),
    ([dict(root="/a", experiment="b"), dict(experiment="c")], dict()),                  # nested contexts
    ([dict(root="/a", experiment="b")], dict(root="/ignored", experiment="ignored")),   # Run() wins
    ([dict(root="/a", experiment="b")], dict(index_root="/also/ignored")),              # ... even for index_root
    ([dict(index_root="/explicit/root")], dict(total_visible_gpus=0)),
    ([], dict(total_visible_gpus=0)),                                                   # no context at all
]
FLIPR_NQ = (64, 70, 72, 96)


def segmented_inputs():
    """scores [sum(lengths), 33] fp32 and lengths [50] int64 of 50 segments of 1..39 rows."""
    g = torch.Generator().manual_seed(1)
    lengths = torch.randint(1, 40, (50,), generator=g)
    return torch.randn(int(lengths.sum()), 33, generator=g), lengths


def flipr_inputs(nq):
    g = torch.Generator().manual_seed(nq)
    n, nd = 5, 30
    Q0 = torch.nn.functional.normalize(torch.randn(n, nq, 128, generator=g), dim=-1).bfloat16().float()
    D0 = torch.nn.functional.normalize(torch.randn(n, nd, 128, generator=g), dim=-1).bfloat16().float()
    M0 = torch.rand(n, nd, 1, generator=g) > 0.3
    M0[:, 0] = True
    return Q0, D0, M0, torch.linspace(0.5, 1.5, n), torch.tensor([30, 7, 19, 1, 24])


def methods_inputs():
    g = torch.Generator().manual_seed(3)
    B, nway, nq, nd = 3, 2, 40, 24
    Q0 = torch.nn.functional.normalize(torch.randn(B, nq, 128, generator=g), dim=-1).bfloat16().float()
    D0 = torch.nn.functional.normalize(torch.randn(B * nway, nd, 128, generator=g), dim=-1).bfloat16().float()
    M0 = torch.rand(B * nway, nd, 1, generator=g) > 0.3
    M0[:, 0] = True
    return Q0, D0, M0, nway


def methods_run(model, Q0, D0, M0, nway):
    """The three caller shapes of ColBERT.score plus compute_ib_loss_new, values and gradients."""
    B = Q0.size(0)
    Q, D = Q0.clone().requires_grad_(True), D0.clone().requires_grad_(True)
    s = model.score(Q.repeat_interleave(nway, dim=0).contiguous(), D, M0)          # colbert.py:71-73
    loss = model.compute_ib_loss_new(Q, D, M0)                                       # colbert.py:74-78
    (s.sum() + loss).backward()
    out = {"train_scores": s.detach(), "train_loss": loss.detach(), "train_dQ": Q.grad.clone(),
           "train_dD": D.grad.clone()}
    items, imask = D0[:4], M0[:4]                                                    # FLMR_executor.py:826-833
    Qd = Q0.repeat_interleave(4, dim=0).contiguous()
    out["eval"] = model.score(Qd, items.repeat(B, 1, 1), imask.repeat(B, 1, 1)).reshape(B, -1).detach()
    out["one"] = model.score(Q0[:1], D0, M0).detach()                                # colbert.py:282
    return out


def rag_item_embeddings(doclens):
    """pid -> (emb [Nd_max, 128] bf16-exact fp32, mask [Nd_max, 1]) as rag_model_blip.py:303-330 holds them."""
    rng = np.random.default_rng(5)
    nd_max = int(doclens.max())
    items = {}
    for pid, n in enumerate(doclens):
        e = np.zeros((nd_max, 128), dtype=np.float32)
        e[:n] = rng.standard_normal((n, 128)).astype(np.float32)
        e[:n] /= np.linalg.norm(e[:n], axis=1, keepdims=True)
        e = torch.from_numpy(e).bfloat16().float().numpy()
        m = np.zeros((nd_max, 1), dtype=np.float32)
        m[:n] = 1
        items[pid] = (e, m)
    return items


def rag_retrieved_ids(exact_scores, n_docs=3, n_retrieve=5, seed=11):
    """The passages rag_model_blip.py:397-410 keeps: random.sample(n_docs) of each query's top n_retrieve."""
    random.seed(seed)
    top = np.argsort(-exact_scores, axis=1, kind="stable")[:, :n_retrieve]
    return np.array([random.sample(row.tolist(), n_docs) for row in top])


def main(reference):
    sys.path.insert(0, HERE)
    import make_golden
    make_golden.REF = reference
    ColBERTConfig, ColBERT, colbert_score, colbert_score_packed = make_golden.import_reference()[:4]
    from colbert.infra import Run, RunConfig
    out = {}

    # segmented_maxsim.cpp (test_oracle.py)
    scores, lengths = segmented_inputs()
    out["segmented_maxsim"] = ColBERT.segmented_maxsim(scores, lengths).numpy()

    # index addressing: the reference's default root is <cwd at import>/experiments, recorded as "<cwd>"
    cwd = os.getcwd()
    paths = []
    for stack, ckw in PATH_SCENARIOS:
        with contextlib.ExitStack() as es:
            for kw in stack:
                es.enter_context(Run().context(RunConfig(**kw)))
            root = ColBERTConfig.from_existing(ColBERTConfig(**ckw), Run().config).index_root_
            want = os.path.join(root, "temp_index.nbits=8")
            want_abs = os.path.join(root, "/abs/idx")
        paths.append(dict(stack=stack, config=ckw, want=want.replace(cwd, "<cwd>", 1),
                          want_abs=want_abs.replace(cwd, "<cwd>", 1)))
    out["paths_json"] = np.array(json.dumps(paths))

    # interaction='flipr'
    for nq in FLIPR_NQ:
        Q0, D0, M0, w, lens = flipr_inputs(nq)
        cfg = ColBERTConfig(total_visible_gpus=0, interaction="flipr", query_maxlen=64)
        for tag, rows in (("one", slice(0, 1)), ("all", slice(0, Q0.size(0)))):
            Q, D = Q0[rows].clone().requires_grad_(True), D0.clone().requires_grad_(True)
            s = colbert_score(Q, D * M0, M0, config=cfg, use_gpu=False)
            (s * w).sum().backward()
            out["flipr_%d_%s_scores" % (nq, tag)] = s.detach().numpy()
            out["flipr_%d_%s_dQ" % (nq, tag)] = Q.grad.numpy()
            out["flipr_%d_%s_dD" % (nq, tag)] = D.grad.numpy()
        packed = torch.cat([D0[i, :l] for i, l in enumerate(lens)])
        out["flipr_%d_packed" % nq] = colbert_score_packed(Q0[:1], packed, lens, cfg).numpy()

    # ColBERT.score / compute_ib_loss_new as methods
    class _Model:
        colbert_config = ColBERTConfig(total_visible_gpus=0, nway=2, use_ib_negatives=True)
        use_gpu = False
        loss_fn = torch.nn.CrossEntropyLoss()
        score = ColBERT.score
        compute_ib_loss_new = ColBERT.compute_ib_loss_new

    for key, v in methods_run(_Model(), *methods_inputs()).items():
        out["methods_" + key] = v.numpy()

    # the RAG re-score of the retrieved passages (rag_model_blip.py:411-441) and its query gradient
    cs = np.load(os.path.join(HERE, "callsites.npz"))
    items = rag_item_embeddings(cs["doclens"])
    ids = rag_retrieved_ids(cs["exact_scores_bf16"])

    class _Encoder:
        colbert_config = ColBERTConfig(total_visible_gpus=0)
        use_gpu = False
        score = ColBERT.score

    Qr = torch.from_numpy(cs["queries"]).clone().requires_grad_(True)
    want = []
    for b in range(ids.shape[0]):
        E = torch.stack([torch.Tensor(items[i][0]) for i in ids[b]])
        M = torch.stack([torch.Tensor(items[i][1]) for i in ids[b]])
        want.append(_Encoder().score(Qr[[b]].repeat_interleave(ids.shape[1], dim=0).contiguous(), E, M))
    want = torch.stack(want)
    want.sum().backward()
    out["rag_ids"] = ids
    out["rag_scores"] = want.detach().numpy()
    out["rag_dQ"] = Qr.grad.numpy()

    path = os.path.join(HERE, "reference_checks.npz")
    np.savez_compressed(path, **out)
    print("%s (%.1f KB)" % (path, os.path.getsize(path) / 1024))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
