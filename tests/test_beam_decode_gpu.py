"""CTC beam search on the GPU (k_ctc_beam_decode): against the float64 reference in tests/_beam_ref.py, against brute force
where nothing is pruned, against the CTC loss kernel, and end to end with the recogniser."""
import importlib

import numpy as np
import pytest
import torch

import sgan_oracle as O
from _beam_ref import _peaked_logits, ctc_beam_decode, frame_log_probs, labeling_log_probs
from _parity import IN_DIM, _recognizer, na

pytestmark = pytest.mark.gpu
ops = importlib.import_module("scrabble-gan_b200.ops")
abi = importlib.import_module("scrabble-gan_b200._abi")
decode = importlib.import_module("scrabble-gan_b200.decode")

MARGIN = 1e-4          # nats: a pruning decision closer than this may go either way in fp32
TOL_LOGP = 1e-4


def _run(rt, p, il, w, k, merge=True):
    dec, dlen, lp = ops.ctc_beam_decode(rt, p.to(rt.device), None if il is None else il.to(rt.device), w, k, merge)
    return dec.cpu().numpy(), dlen.cpu().numpy(), lp.cpu().numpy()


def _paths(dec, dlen, k, i):
    return dec[k, i, :dlen[k, i]].tolist()


# (B, T, C, beam_width, top_paths) and the floor on the share of samples whose reference margin exceeds MARGIN (observed
# shares: 0.805, 0.984, 1, 0.125, 1).  At beam_width 100 and 128 over thousands of candidates per frame, a gap below 1e-4
# nats between the last kept and the first pruned total somewhere in 39 or 300 frames is common, so the share of strictly
# checked samples cannot reach 99 % there; every sample is compared, and at least 99 % must agree exactly.
REFERENCE_CASES = [(256, 39, 81, 100, 1, 0.75), (64, 59, 53, 16, 4, 0.95), (33, 1, 2, 8, 2, 1.0), (16, 300, 81, 128, 3, 0.12),
                   (512, 19, 53, 1, 1, 0.99)]


@pytest.mark.parametrize("b,t,c,w,k,qualify", REFERENCE_CASES)
def test_beam_decode_matches_reference(rt, b, t, c, w, k, qualify):
    """Paths equal the reference wherever its margin exceeds MARGIN (a near-tie there may resolve either way in fp32), at
    least `qualify` of the samples have such a margin, at least 99 % of all samples agree, and log_prob agrees to TOL_LOGP
    wherever the paths do."""
    p = torch.softmax(_peaked_logits(b * 1000 + t, b, t, c), -1)
    g = torch.Generator().manual_seed(b + t)
    il = torch.randint(0, t + 1, (b,), generator=g).int()
    il[:2] = torch.tensor([0, t])[:min(2, b)]
    dec, dlen, lp = _run(rt, p, il, w, k)
    exp, exp_lp, margin = ctc_beam_decode(p.numpy(), il.numpy(), w, k)
    assert np.all(dec[np.arange(t)[None, None, :] >= dlen[..., None]] == -1), "padding"
    agree = 0
    for i in range(b):
        same = all(_paths(dec, dlen, j, i) == exp[j][i] for j in range(k))
        if margin[i] > MARGIN:
            assert same, "sample {} (margin {:.2e}): {} vs reference {}".format(
                i, margin[i], [_paths(dec, dlen, j, i) for j in range(k)], [exp[j][i] for j in range(k)])
        if same:
            agree += 1
            fin = np.isfinite(exp_lp[i])
            assert np.array_equal(np.isfinite(lp[i]), fin)
            assert np.all(np.abs(lp[i][fin] - exp_lp[i][fin]) <= TOL_LOGP), (i, lp[i], exp_lp[i])
    share = float(np.mean(margin > MARGIN))
    print("qualifying {:.3f}, agreeing {:.4f}".format(share, agree / b))
    assert share >= qualify, "only {:.3f} of the samples are checked strictly".format(share)
    assert agree >= 0.99 * b, (agree, b)


@pytest.mark.parametrize("c,t", [(3, 6), (4, 4), (2, 6)])
def test_beam_decode_exact_without_pruning(rt, c, t):
    """beam_width covers every prefix: path j is the j-th most probable labeling, scored log p(labeling | x)."""
    g = torch.Generator().manual_seed(7 * c + t)
    p = torch.softmax(torch.randn(6, t, c, generator=g) * 1.5, -1)
    dec, dlen, lp = _run(rt, p, None, 128, 5, merge=False)
    x = frame_log_probs(p.numpy())
    for i in range(6):
        exact = sorted(labeling_log_probs(x[i]).items(), key=lambda kv: -kv[1])
        for j in range(5):
            if j >= len(exact):                                  # fewer labelings of positive probability than paths
                assert dlen[j, i] == 0 and np.isneginf(lp[i, j]), (i, j)
                continue
            assert tuple(_paths(dec, dlen, j, i)) == exact[j][0], (i, j)
            assert abs(lp[i, j] - exact[j][1]) <= TOL_LOGP, (i, j, lp[i, j], exact[j][1])


@pytest.mark.parametrize("b,t,c,w", [(64, 39, 81, 16), (8, 6, 3, 128)])
def test_beam_score_bounded_by_ctc_loss(rt, b, t, c, w):
    """Path 0's log_prob (merge_repeated=False) is the probability of its labeling over the alignments the beam kept: at
    most -CTC loss of that labeling, equal to it when nothing is pruned (the second case).  The loss kernel applies the
    softmax itself, so it gets the logits the probabilities were made from."""
    z = _peaked_logits(5 + t, b, t, c) if c > 3 else torch.randn(b, t, c, generator=torch.Generator().manual_seed(5)) * 1.5
    zd = z.to(rt.device)
    p = ops.softmax_rows(rt, zd)
    il = torch.full((b,), t, dtype=torch.int32, device=rt.device)
    dec, dlen, lp = ops.ctc_beam_decode(rt, p, il, w, 1, False)
    labels = dec[0].clamp_min(0).contiguous()
    loss, _ = ops.ctc(rt, zd, labels, want_grad=False, input_length=il, label_length=dlen[0].contiguous())
    got, bound = lp[:, 0].cpu().numpy().astype(np.float64), -loss.cpu().numpy().astype(np.float64)
    assert np.all(got <= bound + TOL_LOGP), np.max(got - bound)
    if c == 3:                                                   # 1 + 2 + ... + 2^6 = 127 prefixes <= 128: nothing pruned
        assert np.all(np.abs(got - bound) <= TOL_LOGP), np.max(np.abs(got - bound))


def test_beam_decode_input_length_is_per_row(rt):
    b, t, c = 24, 39, 53
    p = torch.softmax(_peaked_logits(31, b, t, c), -1)
    il = torch.randint(1, t + 1, (b,), generator=torch.Generator().manual_seed(3)).int()
    dec, dlen, lp = _run(rt, p, il, 32, 3)
    for i in range(b):
        n = int(il[i])
        d1, l1, p1 = _run(rt, p[i:i + 1, :n].contiguous(), None, 32, 3)
        for j in range(3):
            assert _paths(dec, dlen, j, i) == _paths(d1, l1, j, 0), (i, j)
        assert np.array_equal(lp[i], p1[0]), (i, lp[i], p1[0])


def test_beam_decode_is_deterministic(rt):
    p = torch.softmax(_peaked_logits(41, 128, 39, 81), -1).to(rt.device)
    a = ops.ctc_beam_decode(rt, p, None, 100, 4)
    b = ops.ctc_beam_decode(rt, p, None, 100, 4)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_beam_decode_limits(rt):
    p = torch.full((2, 5, 4), 0.25, device=rt.device)
    for w, k in ((0, 1), (129, 1), (4, 5)):
        with pytest.raises(abi.SganError):
            ops.ctc_beam_decode(rt, p, None, w, k)
    with pytest.raises(abi.SganError):
        ops.ctc_beam_decode(rt, torch.full((2, 5, 129), 1 / 129, device=rt.device), None, 4, 1)
    dec, dlen, lp = ops.ctc_beam_decode(rt, p, None, 128, 128)              # the largest beam is accepted
    assert tuple(dec.shape) == (128, 2, 5) and tuple(lp.shape) == (2, 128)


# ----------------------------------------------------------------------------------------------------
# with the recogniser
# ----------------------------------------------------------------------------------------------------
def test_ctc_beam_decode_of_frame_probs(rt):
    rt.set_mode("fp32")
    b, l, classes = 64, 6, 53
    R = _recognizer(rt, O.make_recognizer_params(90, torch.float32, output_classes=classes, bias_scale=0.3), classes)
    g = torch.Generator().manual_seed(91)
    x = torch.rand(b, 32, 16 * l, 1, generator=g) * 2 - 1
    il = torch.randint(1, 4 * l, (b,), generator=g).int()
    probs = R.frame_probs(x)
    decoded, log_prob = decode.ctc_beam_decode(probs, il, beam_width=16, top_paths=2)
    assert len(decoded) == 2 and all(d.dtype == torch.int32 and tuple(d.shape) == (b, 4 * l - 1) for d in decoded)
    assert tuple(log_prob.shape) == (b, 2)
    exp, exp_lp, margin = ctc_beam_decode(probs, il.numpy(), 16, 2)
    agree = 0
    for i in range(b):
        got = [[v for v in decoded[j][i].tolist() if v >= 0] for j in range(2)]
        same = got == [exp[0][i], exp[1][i]]
        assert same or margin[i] <= MARGIN, (i, got, exp[0][i], exp[1][i])
        agree += same
        if same:
            assert np.all(np.abs(log_prob[i].cpu().numpy() - exp_lp[i]) <= TOL_LOGP)
    assert agree >= 0.95 * b, agree


def test_evaluate_recognizer_with_beam(rt):
    rt.set_mode("fp32")
    classes = 53
    R = _recognizer(rt, O.make_recognizer_params(95, torch.float32, output_classes=classes, bias_scale=0.3), classes)
    g = torch.Generator().manual_seed(96)
    batches = [(torch.rand(b, 32, 16 * l, 1, generator=g) * 2 - 1, torch.randint(0, classes - 1, (b, l), generator=g))
               for b, l in ((32, 3), (16, 7))]
    b, l = 12, 5
    lens = torch.randint(1, l + 1, (b,), generator=g)
    batches.append((torch.rand(b, 32, 16 * l, 1, generator=g) * 2 - 1, torch.randint(0, classes - 1, (b, l), generator=g),
                    4 * lens - 1, lens))
    greedy = decode.evaluate_recognizer(R, iter(batches))
    n0 = rt.launch_count()
    again = decode.evaluate_recognizer(R, iter(batches), beam_width=None)
    n_none = rt.launch_count() - n0
    n0 = rt.launch_count()
    decode.evaluate_recognizer(R, iter(batches))
    assert again == greedy and rt.launch_count() - n0 == n_none, "beam_width=None must be the greedy path"
    got = decode.evaluate_recognizer(R, iter(batches), beam_width=16)
    d, chars, exact = 0, 0, 0
    for batch in batches:                                        # the composition of the public pieces
        il = batch[2] if len(batch) > 2 else None
        (dec,), _ = decode.ctc_beam_decode(R.frame_probs(batch[0]), il, beam_width=16)
        ll = batch[3] if len(batch) > 3 else torch.full((batch[1].shape[0],), batch[1].shape[1])
        dist = decode.edit_distance(dec, batch[1], None, ll).cpu().numpy()
        d, chars, exact = d + int(dist.sum()), chars + int(ll.sum()), exact + int((dist == 0).sum())
    words = sum(bt[0].shape[0] for bt in batches)
    assert got == {"cer": d / chars, "word_accuracy": exact / words, "words": words, "chars": chars}, got


def test_evaluate_generated_words_with_beam(rt):
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
    out = decode.evaluate_generated_words(G, R, labels, noise=z, beam_width=8)
    imgs = G([z.to(rt.device), torch.from_numpy(labels).to(rt.device)], training=False, ragged=True)
    (dec,), _ = decode.ctc_beam_decode(R.frame_probs(imgs), torch.tensor([4 * n - 1 for n in lens]), beam_width=8)
    assert torch.equal(out["decoded"], dec)
    assert out["words"] == 7 and out["chars"] == sum(lens)
    greedy = decode.evaluate_generated_words(G, R, labels, noise=z)
    none = decode.evaluate_generated_words(G, R, labels, noise=z, beam_width=None)
    assert torch.equal(greedy.pop("decoded"), none.pop("decoded")) and greedy == none
