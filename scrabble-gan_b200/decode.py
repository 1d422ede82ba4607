"""Reading words back with the recogniser: greedy CTC decoding, edit distance, and the character error rate (CER) / word
accuracy of R on real word images or on the generator's own words.

Conventions (those of the CTC loss, csrc/ctc.cu): the blank is the LAST class (C - 1); decoded words and label matrices are
int32 rows padded with -1 on the right; the decoding score is Keras' log_prob, the NEGATIVE sum over frames of
log(max_c p + 1e-7) [TF-SEMANTICS: K.ctc_decode feeds log(y_pred + 1e-7) to tf.nn.ctc_greedy_decoder, whose score is the
negated sum of the per-frame maxima].

The probabilities, argmax, decoding and distances are libsgan kernels; torch only allocates and copies.  There is no host
fallback: without a GPU every call raises SganError."""
from __future__ import annotations

import torch

from . import ops
from .bigacgan.net_architecture import to_device_f32, to_device_i32
from .runtime import get_runtime


def ctc_decode(y_pred, input_length, greedy=True, beam_width=100, top_paths=1):
    """tf.keras.backend.ctc_decode.  y_pred: (B, T, C) softmax probabilities (torch tensor, host buffer or DLPack producer);
    input_length: (B,) frames per sample, or None for all T.  Returns ([decoded], log_prob): decoded (B, T) int32 on the
    device, padded with -1 (TF returns int64 and pads only to the longest decoded word), log_prob (B, 1) fp32.  Only greedy
    decoding exists: greedy=False raises NotImplementedError (beam_width and top_paths are accepted for the signature)."""
    if not greedy:
        raise NotImplementedError("ctc_decode: only greedy decoding is implemented")
    rt = get_runtime()
    probs = to_device_f32(rt, y_pred)
    il = None if input_length is None else to_device_i32(rt, input_length).reshape(-1)
    decoded, _, score = ops.ctc_greedy_decode(rt, probs, il)
    return [decoded], score.view(-1, 1)


def edit_distance(hyp, ref, hyp_length=None, ref_length=None):
    """Levenshtein distance between the rows of hyp (B, Lh) and ref (B, Lr <= 64), int32 (B,) on the device
    (tf.edit_distance with normalize=False).  Without a length, a row ends at its first negative entry."""
    rt = get_runtime()
    h, r = to_device_i32(rt, hyp), to_device_i32(rt, ref)
    hl = None if hyp_length is None else to_device_i32(rt, hyp_length).reshape(-1)
    rl = None if ref_length is None else to_device_i32(rt, ref_length).reshape(-1)
    return ops.edit_distance(rt, h, r, hl, rl)


def _read(rt, recognizer, images, labels, input_length, label_length, totals):
    """R's reading of a batch, its distances to the labels added to the device totals; returns the decoded words."""
    probs = recognizer.frame_probs(images)
    decoded, dlen, _ = ops.ctc_greedy_decode(rt, probs, input_length)
    ops.edit_distance(rt, decoded, labels, dlen, label_length, totals)
    return decoded


def _scores(totals) -> dict:
    dist, chars, exact, words = (int(v) for v in totals.cpu().tolist())
    return {"cer": dist / chars if chars else float("nan"), "word_accuracy": exact / words if words else float("nan"),
            "words": words, "chars": chars}


def evaluate_recognizer(recognizer, batches) -> dict:
    """CER (sum of edit distances / sum of reference lengths) and word accuracy of R over `batches`, which yields
    (images, labels) like load_prepare_data -- one length bucket per batch, T = W/4 - 1 frames -- or ragged
    (images, labels, input_length, label_length).  The totals stay on the device: one device-to-host copy at the end.
    Returns {"cer", "word_accuracy", "words", "chars"}."""
    rt = recognizer.rt
    totals = torch.zeros(4, device=rt.device, dtype=torch.int64)
    for batch in batches:
        images, labels = batch[0], batch[1]
        il = to_device_i32(rt, batch[2]).reshape(-1) if len(batch) > 2 and batch[2] is not None else None
        ll = to_device_i32(rt, batch[3]).reshape(-1) if len(batch) > 3 and batch[3] is not None else None
        _read(rt, recognizer, images, to_device_i32(rt, labels), il, ll, totals)
    return _scores(totals)


def evaluate_generated_words(generator, recognizer, labels, noise=None) -> dict:
    """Generate the words `labels` ((B, L_max) padded with -1) in ONE ragged inference call of G, and let R read them back
    with input_length = 4 len - 1 (the reference R's interface).  noise: z (B, latent_dim), or None to draw it with
    ops.random_.  Returns evaluate_recognizer's dict plus "decoded", R's words (B, 4 L_max - 1) int32 padded with -1."""
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
    decoded = _read(rt, recognizer, images, y, 4 * lens - 1, lens, totals)
    out = _scores(totals)
    out["decoded"] = decoded
    return out


def to_strings(decoded, char_vector):
    """Host helper: rows of class indices (padded with -1) -> list of str through char_vector."""
    rows = decoded.cpu().tolist() if isinstance(decoded, torch.Tensor) else [list(r) for r in decoded]
    return ["".join(char_vector[i] for i in row if 0 <= i < len(char_vector)) for row in rows]
