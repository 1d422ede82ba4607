"""Plain-Python (numpy, float64) restatement of k_ctc_lexicon_scores (csrc/ctc.cu), the yardstick of the lexicon decoder
(tests only): the CTC forward (alpha) recursion of every lexicon word over one sample's frames, vectorised over the words.

Per frame the input is log-softmax(log(p + 1e-7)) over the C classes (_beam_ref.frame_log_probs), blank = C - 1, so a score
is minus K.ctc_batch_cost of the (sample, word) pair [TF-SEMANTICS].  A word holding a symbol outside [0, C - 1) scores -inf;
over no frames the empty word scores 0 and every other word -inf."""
import numpy as np
import torch

from _beam_ref import frame_log_probs


def word_lengths(lexicon):
    """The run of leading entries >= 0 of every row (ops.label_lengths)."""
    lex = np.asarray(lexicon)
    neg = np.concatenate([lex < 0, np.ones((lex.shape[0], 1), bool)], axis=1)
    return neg.argmax(1)


def word_log_probs(x, lexicon, lengths=None):
    """x (T, C) per-frame log-probabilities, lexicon (V, Lmax) padded with -1, lengths (V,) or None (leading entries >= 0).
    Returns (V,) float64: log p(word | x), -inf where the word has no alignment."""
    t_len, c_num = x.shape
    blank = c_num - 1
    lex = np.asarray(lexicon, np.int64)
    v, l_max = lex.shape
    lens = word_lengths(lex) if lengths is None else np.clip(np.asarray(lengths, np.int64), 0, l_max)
    inside = np.arange(l_max)[None, :] < lens[:, None]
    bad = np.any(inside & ((lex < 0) | (lex >= blank)), axis=1)
    if t_len == 0:
        return np.where((lens == 0) & ~bad, 0.0, -np.inf)
    s_max = 2 * l_max + 1
    ext = np.full((v, s_max), blank)
    ext[:, 1::2] = np.where(inside & ~bad[:, None], lex, blank)
    n_states = 2 * lens + 1
    live = np.arange(s_max)[None, :] < n_states[:, None]
    skip = np.zeros((v, s_max), bool)
    skip[:, 3::2] = ext[:, 3::2] != ext[:, 1:-2:2]                    # letter differs from the one before it
    em = x[:, ext]                                                    # (T, V, S)
    alpha = np.full((v, s_max), -np.inf)
    alpha[:, :2] = em[0, :, :2]
    alpha[~live] = -np.inf
    for t in range(1, t_len):
        a1 = np.concatenate([np.full((v, 1), -np.inf), alpha[:, :-1]], axis=1)
        a2 = np.concatenate([np.full((v, 2), -np.inf), alpha[:, :-2]], axis=1)[:, :s_max]
        a2 = np.where(skip, a2, -np.inf)
        alpha = np.logaddexp(np.logaddexp(alpha, a1), a2) + em[t]
        alpha[~live] = -np.inf
    rows = np.arange(v)
    last = alpha[rows, n_states - 1]
    prev = np.where(n_states >= 2, alpha[rows, np.maximum(n_states - 2, 0)], -np.inf)
    out = np.logaddexp(last, prev)
    out[bad] = -np.inf
    return out


def lexicon_scores(probs, input_length, lexicon):
    """k_ctc_lexicon_scores restated: probs (B, T, C) softmax probabilities, input_length (B,) frames (clamped to [0, T]) or
    None, lexicon (V, Lmax) padded with -1.  Returns (B, V) float64."""
    p = np.asarray(probs.detach().cpu() if isinstance(probs, torch.Tensor) else probs)
    b, t_max, _ = p.shape
    x = frame_log_probs(p)
    lex = np.asarray(lexicon)
    lens = word_lengths(lex)
    out = np.empty((b, lex.shape[0]))
    for i in range(b):
        t_b = t_max if input_length is None else min(max(int(np.asarray(input_length).reshape(-1)[i]), 0), t_max)
        out[i] = word_log_probs(x[i, :t_b], lex, lens)
    return out
