"""Known-answer tests of the CTC beam-search reference in tests/_beam_ref.py, and the GPU-only guarantee of
decode.ctc_beam_decode."""
import importlib
import math

import numpy as np
import pytest

from _beam_ref import beam_decode_one, ctc_beam_decode, frame_log_probs, labeling_log_probs

abi = importlib.import_module("scrabble-gan_b200._abi")


def _random_probs(rng, t, c):
    return rng.dirichlet(np.full(c, 0.7), size=(1, t)).astype(np.float32)


@pytest.mark.parametrize("c,t", [(2, 6), (3, 6), (4, 5), (4, 6)])
def test_exact_without_pruning(c, t):
    """Nothing pruned: path k is the k-th most probable labeling and its score is log p(labeling | x)."""
    rng = np.random.default_rng(10 * c + t)
    for _ in range(3):
        p = _random_probs(rng, t, c)
        x = frame_log_probs(p)[0]
        exact = sorted(labeling_log_probs(x).items(), key=lambda kv: -kv[1])
        k = min(6, len(exact))
        paths, scores, margin = beam_decode_one(x, 10 ** 6, k, merge_repeated=False)
        assert margin > 0
        for j in range(k):
            assert tuple(paths[j]) == exact[j][0], (j, paths[j], exact[j])
            assert abs(scores[j] - exact[j][1]) <= 1e-9, (j, scores[j], exact[j][1])


def test_input_transform_is_log_softmax_of_log_p_plus_eps():
    p = np.array([[[0.5, 0.25, 0.25, 0.0]]], np.float32)            # sums to 1 exactly: (p + eps) / (1 + C eps)
    x = frame_log_probs(p)[0, 0]
    q = (p[0, 0].astype(np.float64) + 1e-7) / (1 + 4e-7)
    assert np.allclose(x, np.log(q), rtol=0, atol=1e-12)


def _onehotish(frames, c, hi=0.97):
    p = np.full((1, len(frames), c), (1 - hi) / (c - 1), np.float32)
    for t, k in enumerate(frames):
        p[0, t, k] = hi
    return p


def test_merge_repeated_quirk():
    """a, blank, a is the prefix "a a"; TF v1 writes it out merged as "a" [TF-SEMANTICS]; the score is the prefix's either way."""
    a, blank = 0, 2
    p = _onehotish([a, blank, a], 3)
    (merged,), s_merged, _ = ctc_beam_decode(p, None, beam_width=8, top_paths=1, merge_repeated=True)
    (plain,), s_plain, _ = ctc_beam_decode(p, None, beam_width=8, top_paths=1, merge_repeated=False)
    assert plain == [[a, a]] and merged == [[a]]
    assert s_merged[0, 0] == s_plain[0, 0]
    exact = labeling_log_probs(frame_log_probs(p)[0])
    assert abs(s_plain[0, 0] - exact[(a, a)]) <= 1e-9             # nothing pruned at this width


def test_empty_input_and_paths_beyond_the_live_beams():
    p = _onehotish([0, 1], 3)
    paths, scores, _ = ctc_beam_decode(p, np.array([0]), beam_width=4, top_paths=3)
    assert [paths[k][0] for k in range(3)] == [[], [], []]
    assert scores[0, 0] == 0.0 and math.isinf(scores[0, 1]) and scores[0, 1] < 0 and math.isinf(scores[0, 2])
    # one frame of C = 2: two live beams (the empty word and "0"), the rest empty with -inf
    p = np.array([[[0.6, 0.4]]], np.float32)
    paths, scores, _ = ctc_beam_decode(p, None, beam_width=8, top_paths=5)
    assert [paths[k][0] for k in range(5)] == [[0], [], [], [], []]
    assert np.all(np.isfinite(scores[0, :2])) and np.all(np.isneginf(scores[0, 2:]))


def test_tie_goes_to_the_lower_index():
    """Two classes of equal probability: with one beam kept, the extension by the lower class wins."""
    p = np.array([[[0.4, 0.4, 0.2]]], np.float32)
    (paths,), _, margin = ctc_beam_decode(p, None, beam_width=1, top_paths=1)
    assert paths == [[0]]
    assert margin[0] > 0                                           # an exact tie is not a near-tie


def test_beam_decode_without_gpu_raises():
    """No host fallback: the public beam decoder needs the GPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    decode = importlib.import_module("scrabble-gan_b200.decode")
    with pytest.raises(abi.SganError):
        decode.ctc_beam_decode(_onehotish([0, 1], 3), None, beam_width=4)
