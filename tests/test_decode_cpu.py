"""Known-answer tests of the decoding reference in tests/_decode_ref.py (greedy CTC decoding, Levenshtein distance) and the
GPU-only guarantee of the public decode module."""
import functools
import importlib
import itertools
import math

import numpy as np
import pytest

from _decode_ref import ctc_greedy_decode, levenshtein

abi = importlib.import_module("scrabble-gan_b200._abi")


def _probs(frames, c):
    """One-hot-ish probabilities: frame t puts 0.9 on class frames[t], the rest spread evenly."""
    p = np.full((1, len(frames), c), 0.1 / (c - 1), dtype=np.float32)
    for t, k in enumerate(frames):
        p[0, t, k] = 0.9
    return p


def test_greedy_merges_repeats_then_drops_blanks():
    a, b, blank = 0, 1, 2
    words, score = ctc_greedy_decode(_probs([a, a, blank, a, b, b], 3))
    assert words == [[a, a, b]]
    assert score[0] == pytest.approx(-6 * math.log(np.float32(0.9) + np.float32(1e-7)), rel=1e-12)


def test_greedy_all_blank_is_the_empty_word():
    words, _ = ctc_greedy_decode(_probs([4] * 7, 5))
    assert words == [[]]


def test_greedy_input_length_truncates():
    p = _probs([0, 2, 1, 2, 3], 5)
    words, score = ctc_greedy_decode(p, np.array([3]))
    assert words == [[0, 2, 1]]
    assert score[0] == pytest.approx(-3 * math.log(np.float32(0.9) + np.float32(1e-7)), rel=1e-12)
    words, score = ctc_greedy_decode(p, np.array([0]))
    assert words == [[]] and score[0] == 0.0


def test_greedy_tie_goes_to_lowest_index():
    p = np.array([[[0.2, 0.4, 0.4, 0.0], [0.4, 0.1, 0.1, 0.4]]], dtype=np.float32)
    words, _ = ctc_greedy_decode(p)
    assert words == [[1, 0]]


def test_levenshtein_kats():
    assert levenshtein("kitten", "sitting") == 3
    assert levenshtein("", "abc") == 3
    assert levenshtein([1, 2], []) == 2
    assert levenshtein([], []) == 0


def test_levenshtein_equals_recursive_definition():
    @functools.lru_cache(maxsize=None)
    def rec(a, b):
        if not a or not b:
            return len(a) + len(b)
        return min(rec(a[1:], b) + 1, rec(a, b[1:]) + 1, rec(a[1:], b[1:]) + (a[0] != b[0]))

    words = ["".join(w) for n in range(5) for w in itertools.product("abc", repeat=n)]
    for a in words:
        for b in words:
            assert levenshtein(a, b) == rec(a, b), (a, b)


def test_decode_without_gpu_raises():
    """No host fallback: the public decoder needs the GPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    decode = importlib.import_module("scrabble-gan_b200.decode")
    with pytest.raises(abi.SganError):
        decode.ctc_decode(_probs([0, 1], 3), None)
    with pytest.raises(abi.SganError):
        decode.edit_distance(np.zeros((1, 2), np.int32), np.zeros((1, 2), np.int32))
    with pytest.raises(NotImplementedError):
        decode.ctc_decode(_probs([0, 1], 3), None, greedy=False)
