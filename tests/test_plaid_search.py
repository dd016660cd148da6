"""oracle/plaid_search.py (restated PLAID CPU search) pinned against the reference's IndexScorer.

tests/golden/plaid_search.npz holds what the unmodified reference returned (candidate pids, centroid
scores, pids surviving filter_pids.cpp, final ranking) — see tests/golden/make_golden_plaid_search.py.
The search tests run the oracle on its restatements of the reference's native kernels and, where
oracle/build_ref.py compiled them into oracle/_ref/, on the compiled kernels as well.
"""
import itertools
import os

import numpy as np
import pytest
import torch

from oracle import plaid_search as P

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "plaid_search.npz")


def _searchers(index):
    """The restated kernels always; the reference's compiled kernels too where they were built."""
    return [P.PlaidSearcher(index, compiled=c) for c in ([False, True] if P.have_reference_kernels() else [False])]


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLDEN)


@pytest.fixture(scope="module")
def index(gold):
    return P.PlaidIndex.from_npz(gold)


def _configs(gold):
    return [(int(a), float(b), int(c), int(d)) for a, b, c, d in gold["configs"]]


def _bf16_bits_to_f32(bits):
    return torch.from_numpy((bits.astype(np.uint32) << 16).view(np.float32).copy())


def test_bit_tables_match_reference_codec(gold, index):
    # residual.py:49-88 for nbits = 2: byte 0b00011011 -> fields 00 01 10 11 -> bit-reversed 00 10 01 11
    assert int(index.reversed_bit_map[0b00011011]) == 0b00100111
    assert index.lut.shape == (256, 4) and index.lut[0b00011011].tolist() == [0, 1, 2, 3]
    for nbits in (1, 2, 4, 8):
        rbm = P.reversed_bit_map(nbits)
        assert sorted(rbm.tolist()) == list(range(256))           # a permutation of byte values
        assert torch.equal(rbm[rbm.long()], torch.arange(256, dtype=torch.uint8))   # and an involution


def test_build_reproduces_reference_index(gold, index):
    """PlaidIndex.build on the original embeddings == what ResidualCodec.compress + optimize_ivf wrote."""
    embs = _bf16_bits_to_f32(gold["embs_bf16"])
    heldout = embs[torch.from_numpy(gold["heldout_idx"])]
    built = P.PlaidIndex.build(embs, gold["doclens"], index.centroids, int(gold["nbits"]), heldout=heldout)
    assert torch.equal(built.codes, index.codes)
    assert torch.equal(built.residuals, index.residuals)
    assert torch.equal(built.ivf, index.ivf) and torch.equal(built.ivf_lengths, index.ivf_lengths)
    assert torch.allclose(built.bucket_cutoffs, index.bucket_cutoffs, rtol=0, atol=1e-7)
    assert torch.allclose(built.bucket_weights, index.bucket_weights, rtol=0, atol=1e-7)


def test_filter_pids_restatement_matches_reference(gold, index):
    for ci, (ncells, thr, ndocs, qmax) in enumerate(_configs(gold)):
        for qi in range(gold["queries"].shape[0]):
            key = "c%d_q%d_" % (ci, qi)
            cs = gold[key + "cscores"]
            kept = P.filter_pids_np(gold[key + "cand"], cs, index.codes.numpy(), index.doclens.numpy(),
                                    index.offsets.numpy(), cs.max(-1) >= thr, ndocs)
            assert kept.tolist() == gold[key + "kept"].tolist(), key


def test_filter_pids_restatement_rejects_undefined_case(index):
    cs = np.zeros((index.centroids.size(0), 3), dtype=np.float32)
    with pytest.raises(ValueError):
        P.filter_pids_np(np.arange(5), cs, index.codes.numpy(), index.doclens.numpy(), index.offsets.numpy(),
                         np.ones(cs.shape[0], dtype=bool), 8)


def test_retrieve_matches_reference(gold, index):
    Q = torch.from_numpy(gold["queries"])
    for s, (ci, (ncells, thr, ndocs, qmax)) in itertools.product(_searchers(index), enumerate(_configs(gold))):
        for qi in range(Q.size(0)):
            key = "c%d_q%d_" % (ci, qi)
            cand, cs = s.retrieve(Q[qi:qi + 1], ncells, qmax)
            assert cand.tolist() == gold[key + "cand"].tolist(), key
            np.testing.assert_allclose(cs.numpy(), gold[key + "cscores"], rtol=0, atol=1e-6)


def test_rank_matches_reference(gold, index):
    Q = torch.from_numpy(gold["queries"])
    for s, (ci, (ncells, thr, ndocs, qmax)) in itertools.product(_searchers(index), enumerate(_configs(gold))):
        for qi in range(Q.size(0)):
            key = "c%d_q%d_" % (ci, qi)
            pids, scores = s.rank(Q[qi:qi + 1], ncells=ncells, threshold=thr, ndocs=ndocs, query_maxlen=qmax)
            assert pids == gold[key + "pids"].tolist(), key
            np.testing.assert_allclose(np.asarray(scores, dtype=np.float32), gold[key + "scores"], rtol=1e-6, atol=1e-6)
            assert len(pids) == ndocs // 4


def test_rank_is_a_subset_of_exhaustive_scoring(gold, index):
    """PLAID's final scores are exact MaxSim over the DEcompressed index, on a pruned passage set."""
    from oracle import maxsim_oracle as O
    Q = gold["queries"]
    ncells, thr, ndocs, qmax = _configs(gold)[2]
    for s in _searchers(index):
        D = P.decompress(index, torch.arange(index.doclens.numel(), dtype=torch.int32), s.compiled).numpy()
        exact = O.maxsim_scores(Q, D, index.doclens.numpy().astype(np.int32), relu=True)
        for qi in range(Q.shape[0]):
            pids, scores = s.rank(torch.from_numpy(Q[qi:qi + 1]), ncells=ncells, threshold=thr, ndocs=ndocs,
                                  query_maxlen=qmax)
            np.testing.assert_allclose(exact[qi, pids], scores, rtol=2e-6, atol=2e-6)
            assert scores[0] <= exact[qi].max() + 1e-5
