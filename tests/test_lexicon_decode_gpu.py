"""Lexicon decoding on the GPU (k_ctc_lexicon_scores, k_ctc_lexicon_topk): scores against the float64 reference in
tests/_lexicon_ref.py and against the CTC loss kernel, the exact top-k against a host sort of the kernel's own scores, the
beam decoder's score as a lower bound, and end to end with the recogniser."""
import importlib

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

import sgan_oracle as O
from _beam_ref import _peaked_logits
from _lexicon_ref import lexicon_scores, word_lengths
from _parity import IN_DIM, _recognizer, na

pytestmark = pytest.mark.gpu
ops = importlib.import_module("scrabble-gan_b200.ops")
abi = importlib.import_module("scrabble-gan_b200._abi")
decode = importlib.import_module("scrabble-gan_b200.decode")

TOL = 1e-4             # |got - ref| <= TOL * max(1, |ref|) on finite scores
WORD_TILE = 64         # words per CTA of k_ctc_lexicon_scores (LEX_WORDS)


def _lexicon(seed, v, letters, lo, hi, with_empty=True):
    """v words of lo..hi letters drawn from `letters` classes, padded with -1 to hi; row 0 is the empty word."""
    rng = np.random.default_rng(seed)
    lex = np.full((v, max(hi, 1)), -1, np.int32)
    for i in range(v):
        n = int(rng.integers(lo, hi + 1))
        lex[i, :n] = rng.integers(0, letters, n)
    if with_empty:
        lex[0] = -1
    return lex


def _dev(rt, a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(rt.device)


def _scores(rt, p, il, lex):
    lexd = _dev(rt, lex)
    return ops.ctc_lexicon_scores(rt, p.to(rt.device), None if il is None else il.to(rt.device), lexd,
                                  ops.label_lengths(rt, lexd))


def _assert_close(got, ref):
    assert np.array_equal(np.isneginf(got), np.isneginf(ref)), np.argwhere(np.isneginf(got) != np.isneginf(ref))[:5]
    fin = np.isfinite(ref)
    err = np.abs(got[fin] - ref[fin]) / np.maximum(1.0, np.abs(ref[fin]))
    assert err.size == 0 or err.max() <= TOL, err.max()


# (B, T, C, V, longest word); 2000, 500 and 7 are not multiples of the 64-word tile
REFERENCE_CASES = [(64, 39, 81, 2000, 10), (16, 300, 81, 500, 31), (33, 1, 2, 7, 3), (9, 39, 81, 1, 10)]


@pytest.mark.parametrize("b,t,c,v,lmax", REFERENCE_CASES)
def test_lexicon_scores_match_reference(rt, b, t, c, v, lmax):
    assert any(n % WORD_TILE for n in (2000, 500, 7))
    p = torch.softmax(_peaked_logits(b * 1000 + t, b, t, c), -1)
    g = torch.Generator().manual_seed(b + t)
    il = torch.randint(0, t + 1, (b,), generator=g).int()
    il[:2] = torch.tensor([0, t])
    lex = _lexicon(v + lmax, v, c - 1, 0 if v > 1 else 1, lmax, with_empty=v > 1)
    got = _scores(rt, p, il, lex).cpu().numpy().astype(np.float64)
    ref = lexicon_scores(p.numpy(), il.numpy(), lex)
    _assert_close(got, ref)
    assert np.isfinite(ref).any() and (v == 1 or np.isneginf(ref).any())


def test_lexicon_scores_match_ctc_loss(rt):
    """-K.ctc_batch_cost (the loss kernel, which applies the softmax itself) on 16 384 seeded (sample, word) pairs of the
    realistic size B = 256, T = 39, C = 81, V = 10 000."""
    b, t, c, v = 256, 39, 81, 10000
    z = _peaked_logits(123, b, t, c).to(rt.device)
    probs = ops.softmax_rows(rt, z)
    lex = _lexicon(124, v, c - 1, 1, 10)
    lexd = _dev(rt, lex)
    lens = ops.label_lengths(rt, lexd)
    scores = ops.ctc_lexicon_scores(rt, probs, None, lexd, lens)
    rng = np.random.default_rng(125)
    bi, vi = torch.from_numpy(rng.integers(0, b, 16384)).to(rt.device), torch.from_numpy(rng.integers(0, v, 16384)).to(rt.device)
    n = bi.shape[0]
    loss, _ = ops.ctc(rt, z[bi].contiguous(), lexd[vi].clamp_min(0).contiguous(), want_grad=False,
                      input_length=torch.full((n,), t, dtype=torch.int32, device=rt.device), label_length=lens[vi].contiguous())
    got = scores[bi, vi].cpu().numpy().astype(np.float64)
    _assert_close(got, -loss.cpu().numpy().astype(np.float64))


def _host_topk(s, k):
    return np.argsort(-s, axis=1, kind="stable")[:, :k]          # descending, equal scores to the lower index


@pytest.mark.parametrize("k", [1, 5, 128])
def test_lexicon_topk_is_exact(rt, k):
    """Against a stable descending sort of the kernel's own fp32 scores: duplicated words (bit-identical scores, the lower
    row first), samples whose every word is -inf (no frames, and one frame against words of two or more letters)."""
    b, t, c, v = 48, 39, 81, 3000
    p = torch.softmax(_peaked_logits(7 + k, b, t, c), -1)
    rng = np.random.default_rng(8 + k)
    base = _lexicon(9 + k, 600, c - 1, 2, 10, with_empty=False)
    lex = base[rng.integers(0, 600, v)]                          # every word about five times
    il = torch.full((b,), t, dtype=torch.int32)
    il[:3] = torch.tensor([0, 1, 0])
    s = _scores(rt, p, il, lex)
    lexd = _dev(rt, lex)
    lens = ops.label_lengths(rt, lexd)
    dec, dlen, lp, idx = ops.ctc_lexicon_topk(rt, s, lexd, lens, k)
    sh = s.cpu().numpy()
    assert np.all(np.isneginf(sh[:3])) and np.isfinite(sh[3:]).all()
    order = _host_topk(sh, k)
    idx = idx.cpu().numpy()
    assert np.array_equal(idx, order)
    assert np.array_equal(lp.cpu().numpy(), np.take_along_axis(sh, order, 1))
    wl = word_lengths(lex)
    dec, dlen = dec.cpu().numpy(), dlen.cpu().numpy()
    for j in range(k):
        assert np.array_equal(dec[j], lex[order[:, j]]) and np.array_equal(dlen[j], wl[order[:, j]]), j
    dup = [i for i in range(b) for j in range(1, k) if sh[i, order[i, j]] == sh[i, order[i, j - 1]]]
    assert k == 1 or len(dup) > 0, "the lexicon must produce equal scores among the chosen words"


def test_lexicon_input_length_is_per_row(rt):
    """A sample scored over its first T_b frames equals that sample sliced to T_b frames, bit for bit."""
    b, t, c = 12, 39, 53
    p = torch.softmax(_peaked_logits(31, b, t, c), -1)
    il = torch.randint(0, t + 1, (b,), generator=torch.Generator().manual_seed(3)).int()
    lex = _lexicon(32, 300, c - 1, 0, 12)
    s = _scores(rt, p, il, lex).cpu()
    for i in range(b):
        n = max(int(il[i]), 1)
        one = _scores(rt, p[i:i + 1, :n].contiguous(), il[i:i + 1], lex).cpu()
        assert torch.equal(s[i], one[0]), i


def test_lexicon_decode_is_deterministic(rt):
    p = torch.softmax(_peaked_logits(41, 128, 39, 81), -1).to(rt.device)
    lex = decode.encode_words([list(w[w >= 0]) for w in _lexicon(42, 5000, 80, 0, 20)])
    a = decode.ctc_lexicon_scores(p, None, lex)
    b = decode.ctc_lexicon_scores(p, None, lex)
    assert torch.equal(a, b)
    (d1, d2), lp1, i1 = decode.ctc_lexicon_decode(p, None, lex, top_paths=2)
    (e1, e2), lp2, i2 = decode.ctc_lexicon_decode(p, None, lex, top_paths=2)
    assert torch.equal(d1, e1) and torch.equal(d2, e2) and torch.equal(lp1, lp2) and torch.equal(i1, i2)


def test_lexicon_limits(rt):
    p = torch.full((2, 5, 4), 0.25, device=rt.device)
    ok = np.array([[0, 1], [2, -1]], np.int32)
    with pytest.raises(abi.SganError):                           # words of 32 letters
        decode.ctc_lexicon_scores(p, None, np.zeros((1, 32), np.int32))
    with pytest.raises(abi.SganError):                           # 129 classes
        decode.ctc_lexicon_scores(torch.full((2, 5, 129), 1 / 129, device=rt.device), None, ok)
    with pytest.raises(abi.SganError):                           # a frame table beyond 200 KB of shared memory
        decode.ctc_lexicon_scores(torch.full((1, 401, 128), 1 / 128, device=rt.device), None, ok)
    with pytest.raises(abi.SganError):
        decode.ctc_lexicon_scores(torch.full((1, 5, 1), 1.0, device=rt.device), None, ok)
    decode.ctc_lexicon_scores(torch.full((1, 400, 128), 1 / 128, device=rt.device), None, ok)       # the largest table
    assert decode.ctc_lexicon_scores(p, None, np.zeros((1, 31), np.int32)).shape == (2, 1)
    for k in (0, 3):                                             # top_paths in [1, min(V, 128)]
        with pytest.raises(abi.SganError):
            decode.ctc_lexicon_decode(p, None, ok, top_paths=k)
    big = np.zeros((200, 1), np.int32)
    with pytest.raises(abi.SganError):
        decode.ctc_lexicon_decode(p, None, big, top_paths=129)
    decoded, lp, idx = decode.ctc_lexicon_decode(p, None, big, top_paths=128)
    assert len(decoded) == 128 and tuple(lp.shape) == (2, 128) and idx[0].tolist() == list(range(128))
    okd, okl = _dev(rt, ok), torch.tensor([2, 1], dtype=torch.int32, device=rt.device)
    none = torch.empty((0,), dtype=torch.int32, device=rt.device)
    n0 = rt.launch_count()                                       # B = 0 or V = 0: nothing to launch
    assert ops.ctc_lexicon_scores(rt, p[:0], None, okd, okl).shape == (0, 2)
    assert ops.ctc_lexicon_scores(rt, p, None, okd[:0], none).shape == (2, 0)
    dec, dlen, lp, idx = ops.ctc_lexicon_topk(rt, torch.empty((0, 2), device=rt.device), okd, okl, 2)
    assert tuple(dec.shape) == (2, 0, 2) and tuple(lp.shape) == (0, 2)
    assert rt.launch_count() == n0


@pytest.mark.parametrize("b,t,c,w,exact", [(64, 20, 53, 16, False), (8, 6, 3, 128, True)])
def test_beam_path_score_is_a_lower_bound(rt, b, t, c, w, exact):
    """With merge_repeated=False the written path is the beam's own labeling, and its beam log_prob sums the alignments the
    beam kept: at most its lexicon score, equal where nothing is pruned (C = 3 over 6 frames has 127 prefixes <= 128)."""
    z = _peaked_logits(5 + t, b, t, c) if c > 3 else torch.randn(b, t, c, generator=torch.Generator().manual_seed(5)) * 1.5
    p = ops.softmax_rows(rt, z.to(rt.device))
    dec, dlen, lp = ops.ctc_beam_decode(rt, p, None, w, 1, False)
    assert int(dlen.max()) <= 31
    words = dec[0, :, :max(int(dlen.max()), 1)].contiguous()      # sample i's path is word i
    s = ops.ctc_lexicon_scores(rt, p, None, words, dlen[0].contiguous())
    got = torch.diagonal(s).cpu().numpy().astype(np.float64)
    beam = lp[:, 0].cpu().numpy().astype(np.float64)
    assert np.all(beam <= got + TOL * np.maximum(1, np.abs(got))), np.max(beam - got)
    if exact:
        assert np.all(np.abs(beam - got) <= TOL * np.maximum(1, np.abs(got))), np.max(np.abs(beam - got))


# ----------------------------------------------------------------------------------------------------
# with the recogniser
# ----------------------------------------------------------------------------------------------------
def test_ctc_lexicon_decode_of_frame_probs(rt):
    rt.set_mode("fp32")
    b, l, classes = 64, 6, 53
    R = _recognizer(rt, O.make_recognizer_params(90, torch.float32, output_classes=classes, bias_scale=0.3), classes)
    g = torch.Generator().manual_seed(91)
    x = torch.rand(b, 32, 16 * l, 1, generator=g) * 2 - 1
    il = torch.randint(1, 4 * l, (b,), generator=g).int()
    lex = _lexicon(92, 777, classes - 1, 0, 8)
    probs = R.frame_probs(x)
    decoded, log_prob, index = decode.ctc_lexicon_decode(probs, il, lex, top_paths=3)
    assert len(decoded) == 3 and all(d.dtype == torch.int32 and tuple(d.shape) == (b, 8) for d in decoded)
    lexd = _dev(rt, lex)
    lens = ops.label_lengths(rt, lexd)
    s = ops.ctc_lexicon_scores(rt, probs, il.to(rt.device), lexd, lens)
    dec, dlen, lp, idx = ops.ctc_lexicon_topk(rt, s, lexd, lens, 3)
    assert all(torch.equal(decoded[j], dec[j]) for j in range(3))
    assert torch.equal(log_prob, lp) and torch.equal(index, idx)
    assert torch.equal(decode.ctc_lexicon_scores(probs, il, lex), s)
    _assert_close(s.cpu().numpy().astype(np.float64), lexicon_scores(probs, il.numpy(), lex))


def _d2h_copies(fn):
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, sum(e.count for e in prof.key_averages() if "DtoH" in e.key)


def _expected(R, batches, lex):
    d, chars, exact = 0, 0, 0
    for batch in batches:                                        # the composition of the public pieces
        il = batch[2] if len(batch) > 2 else None
        (dec,), _, _ = decode.ctc_lexicon_decode(R.frame_probs(batch[0]), il, lex)
        ll = batch[3] if len(batch) > 3 else torch.full((batch[1].shape[0],), batch[1].shape[1])
        dist = decode.edit_distance(dec, batch[1], None, ll).cpu().numpy()
        d, chars, exact = d + int(dist.sum()), chars + int(ll.sum()), exact + int((dist == 0).sum())
    words = sum(bt[0].shape[0] for bt in batches)
    return {"cer": d / chars, "word_accuracy": exact / words, "words": words, "chars": chars}


def test_evaluate_recognizer_with_lexicon(rt):
    rt.set_mode("fp32")
    classes = 53
    R = _recognizer(rt, O.make_recognizer_params(95, torch.float32, output_classes=classes, bias_scale=0.3), classes)
    g = torch.Generator().manual_seed(96)
    batches = [(torch.rand(b, 32, 16 * l, 1, generator=g) * 2 - 1, torch.randint(0, classes - 1, (b, l), generator=g))
               for b, l in ((32, 3), (16, 7))]
    b, l = 12, 5
    lens = torch.randint(1, l + 1, (b,), generator=g)
    labels = torch.randint(0, classes - 1, (b, l), generator=g)
    labels[torch.arange(l)[None, :] >= lens[:, None]] = -1
    batches.append((torch.rand(b, 32, 16 * l, 1, generator=g) * 2 - 1, labels, 4 * lens - 1, lens))
    truth = [row[row >= 0].tolist() for bt in batches for row in bt[1]]
    lex = decode.encode_words(truth + [w[w >= 0].tolist() for w in _lexicon(97, 400, classes - 1, 1, 7)])
    greedy = decode.evaluate_recognizer(R, iter(batches))
    n0 = rt.launch_count()
    again = decode.evaluate_recognizer(R, iter(batches), lexicon=None)
    n_none = rt.launch_count() - n0
    n0 = rt.launch_count()
    decode.evaluate_recognizer(R, iter(batches))
    assert again == greedy and rt.launch_count() - n0 == n_none, "lexicon=None must be the greedy path"
    got, copies = _d2h_copies(lambda: decode.evaluate_recognizer(R, iter(batches), lexicon=lex))
    assert copies == 1, copies
    assert got == _expected(R, batches, lex), got
    with pytest.raises(ValueError):
        decode.evaluate_recognizer(R, iter(batches), beam_width=8, lexicon=lex)


def test_evaluate_generated_words_with_lexicon(rt):
    rt.set_mode("fp32")
    R = _recognizer(rt, O.make_recognizer_params(97, torch.float32, output_classes=53, bias_scale=0.3), 53)
    G = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, initialise=False)
    G.load_state_dict(O.make_generator_params(98, torch.float32, sigma=0.2, bias_scale=0.05))
    g = torch.Generator().manual_seed(99)
    lens = [6, 1, 3, 2, 6, 4, 5]
    labels = np.full((7, 6), -1, np.int32)
    for i, n in enumerate(lens):
        labels[i, :n] = torch.randint(0, 52, (n,), generator=g).numpy()
    z = torch.randn(7, 128, generator=g)
    lex = decode.encode_words([row[row >= 0] for row in labels] + [[0, 1], [5], [7, 7, 3]])
    out, copies = _d2h_copies(lambda: decode.evaluate_generated_words(G, R, labels, noise=z, lexicon=lex))
    assert copies == 1, copies
    imgs = G([z.to(rt.device), torch.from_numpy(labels).to(rt.device)], training=False, ragged=True)
    (dec,), _, _ = decode.ctc_lexicon_decode(R.frame_probs(imgs), torch.tensor([4 * n - 1 for n in lens]), lex)
    assert torch.equal(out["decoded"], dec)
    dist = decode.edit_distance(dec, labels, None, torch.tensor(lens)).cpu().numpy()
    assert {k: v for k, v in out.items() if k != "decoded"} == {
        "cer": int(dist.sum()) / sum(lens), "word_accuracy": float(np.mean(dist == 0)), "words": 7, "chars": sum(lens)}
    greedy = decode.evaluate_generated_words(G, R, labels, noise=z)
    none = decode.evaluate_generated_words(G, R, labels, noise=z, lexicon=None)
    assert torch.equal(greedy.pop("decoded"), none.pop("decoded")) and greedy == none
