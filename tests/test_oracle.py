"""CPU: pin the oracle (numpy + C restatements) against golden vectors produced by the reference's
own code (tests/golden/make_golden.py, make_golden_reference_checks.py), and against the reference's compiled
segmented_maxsim.cpp (oracle/_ref) when it is present."""
import os
import sys

import numpy as np
import pytest

from helpers import ROOT, c_oracle, c_oracle_scores, golden_names, load_golden
from oracle import maxsim_oracle as O

NAMES = golden_names()


def test_golden_fixtures_exist():
    assert len(NAMES) >= 4, "golden fixtures missing: run tests/golden/make_golden.py in the build container"


@pytest.mark.parametrize("name", NAMES)
def test_numpy_oracle_matches_reference_true_max(name):
    g = load_golden(name)
    got = O.maxsim_scores(g["Q"], g["D"], g["doclens"], relu=False)
    np.testing.assert_allclose(got, g["scores_true_max"], rtol=2e-6, atol=2e-5)


@pytest.mark.parametrize("name", NAMES)
def test_numpy_oracle_matches_reference_relu(name):
    g = load_golden(name)
    got = O.maxsim_scores(g["Q"], g["D"], g["doclens"], relu=True)
    np.testing.assert_allclose(got, g["scores_relu"], rtol=2e-6, atol=2e-5)


@pytest.mark.parametrize("name", NAMES)
def test_reference_function_restatements(name):
    g = load_golden(name)
    Q, D, dl = g["Q"], g["D"], g["doclens"]
    # colbert_score_packed (CPU path) for query 0 == segmented_maxsim(D @ Q0.T)
    np.testing.assert_allclose(O.colbert_score_packed(Q[0:1], D, dl), g["scores_relu"][0], rtol=2e-6, atol=2e-5)
    np.testing.assert_allclose(O.segmented_maxsim(D @ Q[0].T, dl), g["segmented_maxsim_q0"], rtol=2e-6, atol=2e-5)
    # colbert_score / colbert_score_reduce on the padded layout
    off = np.concatenate([[0], np.cumsum(dl)])
    nd = int(dl.max())
    Dp = np.zeros((len(dl), nd, D.shape[1]), np.float32)
    M = np.zeros((len(dl), nd), bool)
    for p in range(len(dl)):
        Dp[p, :dl[p]] = D[off[p]:off[p + 1]]
        M[p, :dl[p]] = True
    np.testing.assert_allclose(O.colbert_score(Q[0:1], Dp, M), g["scores_true_max"][0], rtol=2e-6, atol=2e-5)
    red_in = np.matmul(Dp, Q[0:1].transpose(0, 2, 1))
    np.testing.assert_allclose(O.colbert_score_reduce(red_in, M), g["reduce_q0"], rtol=2e-6, atol=2e-5)


@pytest.mark.parametrize("name", NAMES)
def test_topk_matches_reference_sort(name):
    g = load_golden(name)
    k = g["topk_pids"].shape[1]
    s, p = O.topk(g["scores_true_max"], k)
    assert np.array_equal(p, g["topk_pids"])
    np.testing.assert_array_equal(s, g["topk_scores"])


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("relu", [False, True])
def test_c_oracle_matches_golden(name, relu):
    g = load_golden(name)
    got = c_oracle_scores(g["Q"], g["D"], g["doclens"], relu=relu, nthreads=3)
    np.testing.assert_allclose(got, g["scores_relu" if relu else "scores_true_max"], rtol=3e-6, atol=3e-5)


def test_c_oracle_topk_and_edge_cases():
    L = c_oracle()
    s = np.array([1.0, 3.0, 3.0, -2.0], dtype=np.float32)
    out_s = np.empty(6, np.float32)
    out_p = np.empty(6, np.int64)
    assert L.flmr_oracle_topk(s.ctypes.data, 4, 6, 10, out_s.ctypes.data, out_p.ctypes.data) == 0
    assert out_p.tolist() == [11, 12, 10, 13, -1, -1]          # ties -> lower pid first, padding -1
    assert np.isneginf(out_s[4:]).all()
    ns, npid = O.topk(s, 6, pid_base=10)
    assert npid[0].tolist() == out_p.tolist()


def test_ragged_relu_differs_from_true_max():
    """SURVEY hazard 1: the two reference paths disagree on short docs; the oracle keeps both."""
    g = load_golden("g1_ragged_short")
    assert np.abs(g["scores_true_max"] - g["scores_relu"]).max() > 0.1


def test_zero_query_rows_contribute_zero():
    Q, D, dl = O.synth(20, 16, 1, 32, seed=5, ragged=True)
    Qz = np.concatenate([Q, np.zeros((1, 7, 128), np.float32)], axis=1)
    np.testing.assert_allclose(O.maxsim_scores(Qz, D, dl), O.maxsim_scores(Q, D, dl), rtol=1e-6)


def test_bf16_round_matches_torch():
    import torch
    x = np.random.default_rng(0).standard_normal(4096).astype(np.float32)
    assert np.array_equal(O.bf16_round(x), torch.from_numpy(x).bfloat16().float().numpy())


def test_reference_extension_agrees_when_present():
    """O.segmented_maxsim against what the REFERENCE's own segmented_maxsim.cpp returned
    (tests/golden/make_golden_reference_checks.py), and against the compiled extension itself where
    oracle/build_ref.py built it into oracle/_ref/."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden_reference_checks as G
    z = np.load(os.path.join(ROOT, "tests", "golden", "reference_checks.npz"))
    scores, lengths = G.segmented_inputs()
    got = O.segmented_maxsim(scores.numpy(), lengths.numpy())
    np.testing.assert_allclose(got, z["segmented_maxsim"], rtol=1e-6, atol=1e-5)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import build_ref
    mod = build_ref.load()
    if mod is not None:
        np.testing.assert_allclose(got, mod.segmented_maxsim_cpp(scores, lengths).numpy(), rtol=1e-6, atol=1e-5)


def test_training_path_restatement_matches_reference_autograd():
    """oracle ib_loss_and_grads / maxsim_grads vs tests/golden/train_ib_loss.npz, produced by the reference's
    own compute_ib_loss_new / score and torch autograd (tests/golden/make_golden_train.py)."""
    import os
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "train_ib_loss.npz"))
    f32 = lambda bits: (bits.astype(np.uint32) << 16).view(np.float32)
    Q, D, mask, nway = f32(z["Q_bf16"]), f32(z["D_bf16"]), z["mask"], int(z["nway"])
    loss, dQ, dD, S = O.ib_loss_and_grads(Q, D, mask, nway)
    np.testing.assert_allclose(loss, z["ib_loss"], rtol=2e-6)
    np.testing.assert_allclose(dQ, z["ib_dQ"], rtol=1e-4, atol=2e-7)
    np.testing.assert_allclose(dD, z["ib_dD"], rtol=1e-4, atol=2e-7)
    assert (dD[~mask] == 0).all()
    # aligned scores of the training forward (Q repeat_interleave'd) and their gradients
    rows = np.repeat(np.arange(Q.shape[0]), nway)
    cols = np.arange(D.shape[0])
    np.testing.assert_allclose(S[rows, cols], z["scores"], rtol=2e-6)
    dS = np.zeros_like(S)
    dS[rows, cols] = z["score_weights"]
    _, arg = O.all_pairs_scores(Q, D, mask)
    dQ2, dD2 = O.maxsim_grads(Q, D, arg, dS)
    np.testing.assert_allclose(dQ2, z["score_dQ"], rtol=1e-4, atol=2e-7)
    np.testing.assert_allclose(dD2, z["score_dD"], rtol=1e-4, atol=2e-7)
