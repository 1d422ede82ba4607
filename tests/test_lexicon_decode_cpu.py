"""The float64 lexicon-score reference in tests/_lexicon_ref.py against brute force over all alignments, known answers of
decode.encode_words, and the GPU-only guarantee of the lexicon decoder."""
import importlib
import itertools

import numpy as np
import pytest

from _beam_ref import frame_log_probs, labeling_log_probs
from _lexicon_ref import lexicon_scores, word_lengths, word_log_probs

abi = importlib.import_module("scrabble-gan_b200._abi")
decode = importlib.import_module("scrabble-gan_b200.decode")


def _padded(words):
    out = np.full((len(words), max([1] + [len(w) for w in words])), -1, np.int32)
    for i, w in enumerate(words):
        out[i, :len(w)] = w
    return out


@pytest.mark.parametrize("c,t", [(2, 1), (2, 5), (3, 4), (4, 4), (3, 5)])
def test_reference_equals_brute_force(c, t):
    """Every word of up to t + 1 letters over the c - 1 letters: the recursion equals the sum over all alignments, and is
    -inf exactly for the words no alignment emits (too long, or too many repeated letters for t frames)."""
    rng = np.random.default_rng(10 * c + t)
    p = rng.dirichlet(np.full(c, 0.7), size=(1, t)).astype(np.float32)
    x = frame_log_probs(p)[0]
    exact = labeling_log_probs(x)
    words = [w for n in range(t + 2) for w in itertools.product(range(c - 1), repeat=n)]
    got = word_log_probs(x, _padded(words))
    for w, s in zip(words, got):
        if w in exact:
            assert abs(s - exact[w]) <= 1e-9, (w, s, exact[w])
        else:
            assert np.isneginf(s), (w, s)
    assert () in exact                                            # the empty word is covered
    if t >= 2:                                                    # so is a word that fits by length but not by its repeats
        assert (0,) * t not in exact and np.isneginf(got[words.index((0,) * t)])


def test_reference_edge_cases():
    x = frame_log_probs(np.array([[[0.5, 0.3, 0.2], [0.1, 0.6, 0.3]]], np.float32))[0]
    lex = _padded([[], [0, 0], [0, 1], [2], [1, -1, 0]])        # blank (2) as a letter: invalid; a row ends at its first -1
    got = word_log_probs(x, lex)
    assert word_lengths(lex).tolist() == [0, 2, 2, 1, 1]
    assert np.isneginf(got[1])                                 # "a a" needs a blank between the letters: 3 frames
    assert np.isneginf(got[3])
    exact = labeling_log_probs(x)
    assert abs(got[0] - exact[()]) <= 1e-12 and abs(got[2] - exact[(0, 1)]) <= 1e-12 and abs(got[4] - exact[(1,)]) <= 1e-12
    none = word_log_probs(x[:0], lex)                          # no frames: only the empty word, with probability 1
    assert none[0] == 0.0 and np.all(np.isneginf(none[1:]))
    p = np.stack([np.array([[0.5, 0.3, 0.2], [0.1, 0.6, 0.3]], np.float32)] * 2)
    s = lexicon_scores(p, np.array([2, 0]), lex)
    assert np.array_equal(s[0], got) and np.array_equal(s[1], none)


def test_encode_words_known_answers():
    cv = "abc"
    assert decode.encode_words(["ab", "", "cab"], cv).tolist() == [[0, 1, -1], [-1, -1, -1], [2, 0, 1]]
    assert decode.encode_words([[3, 4], [5], np.array([7, 7, 7])]).tolist() == [[3, 4, -1], [5, -1, -1], [7, 7, 7]]
    random_words = [[[1, 2], [0]], [[2, 2, 1]]]               # data_utils' buckets of int-coded words, flattened
    enc = decode.encode_words([w for bucket in random_words for w in bucket], cv)
    assert enc.dtype == np.int32 and enc.tolist() == [[1, 2, -1], [0, -1, -1], [2, 2, 1]]
    assert decode.encode_words([]).shape == (0, 1)
    assert decode.encode_words(["", ""], cv).tolist() == [[-1], [-1]]
    assert decode.encode_words(["a" * 31], "a").shape == (1, 31)


@pytest.mark.parametrize("words,cv", [(["abd"], "abc"), (["ab"], None), (["a" * 32], "a"), ([[0] * 32], None), ([[0, -1]], None),
                                      ([[0, 3]], "abc")])
def test_encode_words_errors(words, cv):
    with pytest.raises(ValueError):
        decode.encode_words(words, cv)


def test_reader_arguments_exclude_each_other():
    """lexicon and beam_width choose different readers: passing both is an error, before anything runs."""
    with pytest.raises(ValueError):
        decode.evaluate_recognizer(None, iter([]), beam_width=4, lexicon=np.zeros((1, 1), np.int32))
    with pytest.raises(ValueError):
        decode.evaluate_generated_words(None, None, np.zeros((1, 1), np.int32), beam_width=4, lexicon=np.zeros((1, 1), np.int32))


def test_lexicon_decode_without_gpu_raises():
    """No host fallback: the public lexicon scores and decoder need the GPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    p = np.full((1, 3, 3), 1 / 3, np.float32)
    lex = np.array([[0, 1]], np.int32)
    with pytest.raises(abi.SganError):
        decode.ctc_lexicon_scores(p, None, lex)
    with pytest.raises(abi.SganError):
        decode.ctc_lexicon_decode(p, None, lex)
