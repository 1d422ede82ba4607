"""Plain-Python restatements of the decoding functions a Keras user of the reference would call, the yardstick of the
decode kernels (tests only): greedy CTC decoding and the Levenshtein distance."""
import math
from typing import Sequence

import numpy as np
import torch

KERAS_EPS = 1e-7       # K.epsilon()


def ctc_greedy_decode(probs, input_length=None):
    """tf.keras.backend.ctc_decode(greedy=True), i.e. tf.nn.ctc_greedy_decoder(log(probs + 1e-7), merge_repeated=True):
    per frame t < input_length[b] the most probable class (np.argmax: ties -> lowest index), repeats merged, then the blank
    (C-1) dropped.  Returns (list of B int lists, neg_sum_log (B,) float64 = -sum_t log(max_c probs[b,t] + 1e-7)); the score is
    [TF-SEMANTICS] (recalled, not checked against TensorFlow).  probs (B, T, C) array / tensor, compared as given."""
    p = np.asarray(probs.detach().cpu() if isinstance(probs, torch.Tensor) else probs)
    b, t_max, c = p.shape
    words, scores = [], np.zeros(b)
    for i in range(b):
        t_b = t_max if input_length is None else min(max(int(np.asarray(input_length).reshape(-1)[i]), 0), t_max)
        best = [int(np.argmax(p[i, t])) for t in range(t_b)]
        words.append([a for t, a in enumerate(best) if a != c - 1 and (t == 0 or best[t - 1] != a)])
        scores[i] = -sum(math.log(np.float32(p[i, t].max()) + np.float32(KERAS_EPS)) for t in range(t_b))   # fp32 add, as Keras
    return words, scores


def levenshtein(a: Sequence[int], b: Sequence[int]) -> int:
    """Edit distance with unit insert / delete / substitute costs: tf.edit_distance(normalize=False) of two sequences."""
    row = list(range(len(b) + 1))
    for i, x in enumerate(a, 1):
        prev, row[0] = row[:], i
        for j, y in enumerate(b, 1):
            row[j] = min(prev[j] + 1, row[j - 1] + 1, prev[j - 1] + (x != y))
    return row[-1]
