"""Reading words back with the recogniser: greedy, beam-search and lexicon CTC decoding, edit distance, and the character
error rate (CER) / word accuracy of R on real word images or on the generator's own words.

Conventions (those of the CTC loss, csrc/ctc.cu): the blank is the LAST class (C - 1); decoded words and label matrices are
int32 rows padded with -1 on the right; the decoding score is Keras' log_prob, the NEGATIVE sum over frames of
log(max_c p + 1e-7) [TF-SEMANTICS: K.ctc_decode feeds log(y_pred + 1e-7) to tf.nn.ctc_greedy_decoder, whose score is the
negated sum of the per-frame maxima].  The beam decoder's log_prob is the log probability of the decoded beam (prefix
beam search, csrc/ctc.cu k_ctc_beam_decode).  The lexicon decoder reads every image as the word of a closed vocabulary with
the highest CTC likelihood; its log_prob is that likelihood, minus K.ctc_batch_cost of the pair (k_ctc_lexicon_scores).

The probabilities, argmax, decoding and distances are libsgan kernels; torch only allocates and copies.  There is no host
fallback: without a GPU every call raises SganError."""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from .bigacgan.net_architecture import to_device_f32, to_device_i32
from .runtime import get_runtime


def _frame_inputs(y_pred, input_length):
    """The runtime, and (y_pred, input_length) on its device: (B, T, C) fp32 probabilities, (B,) int32 frame counts or None."""
    rt = get_runtime()
    return rt, to_device_f32(rt, y_pred), None if input_length is None else to_device_i32(rt, input_length).reshape(-1)


def ctc_decode(y_pred, input_length, greedy=True, beam_width=100, top_paths=1):
    """tf.keras.backend.ctc_decode.  y_pred: (B, T, C) softmax probabilities (torch tensor, host buffer or DLPack producer);
    input_length: (B,) frames per sample, or None for all T.  Returns ([decoded], log_prob): decoded (B, T) int32 on the
    device, padded with -1 (TF returns int64 and pads only to the longest decoded word), log_prob (B, 1) fp32.  Only greedy
    decoding goes through this function: greedy=False raises NotImplementedError (beam_width and top_paths are accepted for
    the signature); beam search is ctc_beam_decode."""
    if not greedy:
        raise NotImplementedError("ctc_decode: greedy=False is not wired here; use decode.ctc_beam_decode for beam search")
    rt, probs, il = _frame_inputs(y_pred, input_length)
    decoded, _, score = ops.ctc_greedy_decode(rt, probs, il)
    return [decoded], score.view(-1, 1)


def ctc_beam_decode(y_pred, input_length, beam_width=100, top_paths=1, merge_repeated=True):
    """tf.keras.backend.ctc_decode(greedy=False): CTC prefix beam search on the GPU.  y_pred: (B, T, C) softmax probabilities
    (C <= 128), input_length: (B,) frames per sample or None for all T; beam_width in [1, 128], top_paths in [1, beam_width].
    Returns ([decoded_0, ..., decoded_{top_paths-1}], log_prob): decoded_k (B, T) int32 on the device, padded with -1, the
    k-th most probable beam; log_prob (B, top_paths) fp32, -inf where a sample has fewer live beams.  merge_repeated merges
    consecutive equal symbols of the written path, as TF v1 does [TF-SEMANTICS]."""
    rt, probs, il = _frame_inputs(y_pred, input_length)
    decoded, _, log_prob = ops.ctc_beam_decode(rt, probs, il, beam_width, top_paths, merge_repeated)
    return list(decoded.unbind(0)), log_prob


MAX_LEXICON_WORD = 31            # letters per lexicon word: the extended label of a word fits one warp (csrc/ctc.cu)


def encode_words(words, char_vector=None):
    """Host helper: a lexicon as the (V, Lmax) int32 matrix of class indices padded with -1 that the lexicon decoder takes,
    Lmax = the longest word (at least 1).  words: strings, mapped through char_vector (class i = char_vector[i]), or
    sequences of int class indices such as the words of `random_words` (flattened over its buckets).  Raises ValueError on
    a character or index outside char_vector (any negative index), on a string without char_vector, and on a word longer
    than 31 letters."""
    index = None if char_vector is None else {ch: i for i, ch in enumerate(char_vector)}
    rows = []
    for w in words:
        if isinstance(w, str):
            if index is None:
                raise ValueError("encode_words: the string {!r} needs a char_vector".format(w))
            unknown = [ch for ch in w if ch not in index]
            if unknown:
                raise ValueError("encode_words: {!r} has characters outside char_vector: {!r}".format(w, "".join(unknown)))
            row = [index[ch] for ch in w]
        else:
            row = [int(c) for c in (w.tolist() if hasattr(w, "tolist") else w)]
            bad = [c for c in row if c < 0 or (char_vector is not None and c >= len(char_vector))]
            if bad:
                raise ValueError("encode_words: {} has class indices outside char_vector: {}".format(row, bad))
        if len(row) > MAX_LEXICON_WORD:
            raise ValueError("encode_words: {!r} has {} letters; lexicon words have at most {}".format(w, len(row),
                                                                                                     MAX_LEXICON_WORD))
        rows.append(row)
    out = np.full((len(rows), max([1] + [len(r) for r in rows])), -1, np.int32)
    for i, r in enumerate(rows):
        out[i, :len(r)] = r
    return out


def _lexicon(rt, lexicon):
    """The lexicon matrix on the device and its word lengths (ops.label_lengths: the run of leading entries >= 0)."""
    lex = to_device_i32(rt, lexicon)
    return lex, ops.label_lengths(rt, lex)


def _best_words(rt, probs, il, lexicon, top_paths=1):
    """Every sample's top_paths most likely words of lexicon = (matrix, lengths) on the device (ops.ctc_lexicon_topk)."""
    return ops.ctc_lexicon_topk(rt, ops.ctc_lexicon_scores(rt, probs, il, *lexicon), *lexicon, top_paths)


def ctc_lexicon_scores(y_pred, input_length, lexicon):
    """log p(word | image) of every (sample, lexicon word) pair, i.e. -K.ctc_batch_cost of the pair, without building the
    replicated batch: (B, V) fp32 on the device.  y_pred: (B, T, C) softmax probabilities (C <= 128, T * C <= 51 200);
    input_length: (B,) frames per sample or None for all T; lexicon: (V, Lmax <= 31) int32 padded with -1 (encode_words).
    A word that cannot fit in a sample's frames scores -inf.  The scores give posteriors over the lexicon, or can be
    combined with word priors; ops.ctc_lexicon_topk ranks any such (B, V) rows."""
    rt, probs, il = _frame_inputs(y_pred, input_length)
    return ops.ctc_lexicon_scores(rt, probs, il, *_lexicon(rt, lexicon))


def ctc_lexicon_decode(y_pred, input_length, lexicon, top_paths=1):
    """Closed-vocabulary decoding: every sample reads as the lexicon words of highest CTC likelihood.  Arguments as in
    ctc_lexicon_scores; 1 <= top_paths <= min(V, 128).  Returns ([decoded_0, ..., decoded_{top_paths-1}], log_prob, index):
    decoded_k (B, Lmax) int32 on the device, the k-th best word padded with -1; log_prob (B, top_paths) fp32, its score;
    index (B, top_paths) int32, its row in the lexicon.  Equal scores go to the lower row."""
    rt, probs, il = _frame_inputs(y_pred, input_length)
    decoded, _, log_prob, index = _best_words(rt, probs, il, _lexicon(rt, lexicon), top_paths)
    return list(decoded.unbind(0)), log_prob, index


def edit_distance(hyp, ref, hyp_length=None, ref_length=None):
    """Levenshtein distance between the rows of hyp (B, Lh) and ref (B, Lr <= 64), int32 (B,) on the device
    (tf.edit_distance with normalize=False).  Without a length, a row ends at its first negative entry."""
    rt = get_runtime()
    h, r = to_device_i32(rt, hyp), to_device_i32(rt, ref)
    hl = None if hyp_length is None else to_device_i32(rt, hyp_length).reshape(-1)
    rl = None if ref_length is None else to_device_i32(rt, ref_length).reshape(-1)
    return ops.edit_distance(rt, h, r, hl, rl)


def _read(rt, recognizer, images, labels, input_length, label_length, totals, beam_width=None, lexicon=None):
    """R's reading of a batch (greedy, path 0 of a beam search of beam_width, or the best word of `lexicon` = (matrix,
    lengths) on the device), its distances to the labels added to the device totals; returns the decoded words."""
    probs = recognizer.frame_probs(images)
    if lexicon is not None:
        decoded, dlen, _, _ = _best_words(rt, probs, input_length, lexicon)
        decoded, dlen = decoded[0], dlen[0]
    elif beam_width is None:
        decoded, dlen, _ = ops.ctc_greedy_decode(rt, probs, input_length)
    else:
        decoded, dlen, _ = ops.ctc_beam_decode(rt, probs, input_length, beam_width)
        decoded, dlen = decoded[0], dlen[0]
    ops.edit_distance(rt, decoded, labels, dlen, label_length, totals)
    return decoded


def _scores(totals) -> dict:
    dist, chars, exact, words = (int(v) for v in totals.cpu().tolist())
    return {"cer": dist / chars if chars else float("nan"), "word_accuracy": exact / words if words else float("nan"),
            "words": words, "chars": chars}


def _check_reader(beam_width, lexicon):
    if lexicon is not None and beam_width is not None:
        raise ValueError("pass either beam_width (open-vocabulary beam search) or lexicon (closed vocabulary), not both")


def evaluate_recognizer(recognizer, batches, beam_width=None, lexicon=None) -> dict:
    """CER (sum of edit distances / sum of reference lengths) and word accuracy of R over `batches`, which yields
    (images, labels) like load_prepare_data -- one length bucket per batch, T = W/4 - 1 frames -- or ragged
    (images, labels, input_length, label_length).  The totals stay on the device: one device-to-host copy at the end.
    beam_width: None reads greedily; an integer reads path 0 of a beam search that wide.  lexicon: a (V, Lmax <= 31) word
    matrix padded with -1 (encode_words): every image reads as its most likely lexicon word (closed vocabulary); it
    excludes beam_width.  Returns {"cer", "word_accuracy", "words", "chars"}."""
    _check_reader(beam_width, lexicon)
    rt = recognizer.rt
    lex = None if lexicon is None else _lexicon(rt, lexicon)
    totals = torch.zeros(4, device=rt.device, dtype=torch.int64)
    for batch in batches:
        images, labels = batch[0], batch[1]
        il = to_device_i32(rt, batch[2]).reshape(-1) if len(batch) > 2 and batch[2] is not None else None
        ll = to_device_i32(rt, batch[3]).reshape(-1) if len(batch) > 3 and batch[3] is not None else None
        _read(rt, recognizer, images, to_device_i32(rt, labels), il, ll, totals, beam_width, lex)
    return _scores(totals)


def evaluate_generated_words(generator, recognizer, labels, noise=None, beam_width=None, lexicon=None) -> dict:
    """Generate the words `labels` ((B, L_max) padded with -1) in ONE ragged inference call of G, and let R read them back
    with input_length = 4 len - 1 (the reference R's interface).  noise: z (B, latent_dim), or None to draw it with
    ops.random_.  beam_width and lexicon as in evaluate_recognizer.  Returns evaluate_recognizer's dict plus "decoded", R's
    words (B, 4 L_max - 1) int32 padded with -1 -- (B, Lmax) of the lexicon with a lexicon."""
    _check_reader(beam_width, lexicon)
    rt = generator.rt
    y = to_device_i32(rt, labels)
    if noise is None:
        if generator.style is not None:
            raise ValueError("a style-encoder generator needs its style images as `noise`")
        z = ops.random_(rt, rt.empty((y.shape[0], generator.latent_dim)))
    else:
        z = to_device_f32(rt, noise)
    images = generator([z, y], training=False, ragged=True)
    lens = ops.label_lengths(rt, y)
    totals = torch.zeros(4, device=rt.device, dtype=torch.int64)
    lex = None if lexicon is None else _lexicon(rt, lexicon)
    decoded = _read(rt, recognizer, images, y, 4 * lens - 1, lens, totals, beam_width, lex)
    out = _scores(totals)
    out["decoded"] = decoded
    return out


def to_strings(decoded, char_vector):
    """Host helper: rows of class indices (padded with -1) -> list of str through char_vector."""
    rows = decoded.cpu().tolist() if isinstance(decoded, torch.Tensor) else [list(r) for r in decoded]
    return ["".join(char_vector[i] for i in row if 0 <= i < len(char_vector)) for row in rows]
