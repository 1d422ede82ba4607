"""Reading words back with the recogniser on the GPU: the three kernels (row softmax, greedy CTC decoding, edit distance)
against the oracle, Recognizer.frame_probs against the CRNN oracle, and the public decode module end to end."""
import importlib

import numpy as np
import pytest
import torch

import sgan_oracle as O
from _decode_ref import ctc_greedy_decode, levenshtein
from _parity import IN_DIM, na, rel_elementwise, rel_max

pytestmark = pytest.mark.gpu
ops = importlib.import_module("scrabble-gan_b200.ops")
abi = importlib.import_module("scrabble-gan_b200._abi")
decode = importlib.import_module("scrabble-gan_b200.decode")

TOL_BF16 = 1e-2            # bf16 TOL_OUT of test_parity_benchpath_gpu.py


def _padded(words, width):
    out = np.full((len(words), width), -1, dtype=np.int32)
    for i, w in enumerate(words):
        out[i, :len(w)] = w
    return out


def _assert_scores_close(got, exp, tol=1e-6):
    got, exp = np.asarray(got, np.float64), np.asarray(exp, np.float64)
    bad = np.abs(got - exp) > tol * np.abs(exp)
    assert not bad.any(), "scores beyond {:.0e} relative at {}: {} vs {}".format(tol, np.nonzero(bad)[0][:5], got[bad][:5], exp[bad][:5])


# ----------------------------------------------------------------------------------------------------
# kernels
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [2, 53, 81, 200])
def test_softmax_rows(rt, c):
    g = torch.Generator().manual_seed(c)
    x = torch.randn(777, c, generator=g) * 3
    y = ops.softmax_rows(rt, x.to(rt.device))
    exp = torch.softmax(x.double(), dim=-1)
    d = (y.double().cpu() - exp).abs()
    # relative to the row's largest probability: an entry e^-18 below it carries the fp32 rounding of z - max (~1e-6 of itself)
    row = float((d.max(-1).values / exp.max(-1).values).max())
    elem = float((d / exp).max())
    assert row <= 1e-6 and elem <= 4e-6, "softmax rows of {}: rel err {:.3e} (row), {:.3e} (element)".format(c, row, elem)


def _decode_case(seed, b, t, c):
    """Per-frame probabilities that follow a planted path: letters repeated over several frames, repeats across and not across
    blanks, all-blank samples, and exact ties for the best class on ~10 % of the frames."""
    g = torch.Generator().manual_seed(seed)
    blank = c - 1
    path = torch.empty(b, t, dtype=torch.long)
    for i in range(b):
        prev = blank
        for s in range(t):
            u = float(torch.rand(1, generator=g))
            prev = prev if u < 0.45 else (blank if u < 0.7 else int(torch.randint(0, c, (1,), generator=g)))
            path[i, s] = prev
    path[0] = blank                                               # all-blank sample
    p = torch.rand(b, t, c, generator=g) * 0.5
    p.scatter_add_(2, path.unsqueeze(-1), torch.ones(b, t, 1))
    tie = torch.rand(b, t, generator=g) < 0.1
    j = torch.randint(0, c, (b, t), generator=g)
    mx = p.max(-1).values
    p[tie, j[tie]] = mx[tie]
    p = p / p.sum(-1, keepdim=True)                               # equal entries stay equal
    il = torch.randint(0, t + 1, (b,), generator=g)
    il[:3] = torch.tensor([0, 1, t])[:min(3, b)]
    return p.float(), il.int()


@pytest.mark.parametrize("b,t,c", [(512, 39, 81), (64, 59, 53), (300, 1, 2), (33, 39, 2), (16, 300, 81), (128, 300, 53)])
def test_ctc_greedy_decode_matches_reference(rt, b, t, c):
    p, il = _decode_case(b * 1000 + t, b, t, c)
    pd = p.to(rt.device)
    for lens in (il, None):
        ild = lens.to(rt.device) if lens is not None else None
        dec, dlen, score = ops.ctc_greedy_decode(rt, pd, ild)
        words, exp_score = ctc_greedy_decode(p, lens.numpy() if lens is not None else None)
        assert np.array_equal(dec.cpu().numpy(), _padded(words, t)), "decoded words differ from the reference"
        assert dlen.cpu().tolist() == [len(w) for w in words]
        _assert_scores_close(score.cpu().numpy(), exp_score)
        dec2, dlen2, score2 = ops.ctc_greedy_decode(rt, pd, ild)
        assert torch.equal(dec, dec2) and torch.equal(dlen, dlen2) and torch.equal(score, score2), "decoding is not repeatable"


def _edit_case(seed, b, hw, rw, alphabet):
    g = np.random.default_rng(seed)
    hl, rl = g.integers(0, hw + 1, b), g.integers(0, rw + 1, b)
    hl[:4], rl[:4] = [0, hw, 0, hw], [rw, 0, 0, rw]
    hyp = g.integers(0, alphabet, (b, hw)).astype(np.int32)
    ref = g.integers(0, alphabet, (b, rw)).astype(np.int32)
    ref[5, :rl[5]] = hyp[5, :rl[5]]
    hl[5] = rl[5]                                                 # an exact match
    exp = np.array([levenshtein(hyp[i, :hl[i]].tolist(), ref[i, :rl[i]].tolist()) for i in range(b)], dtype=np.int32)
    return hyp, ref, hl.astype(np.int32), rl.astype(np.int32), exp


@pytest.mark.parametrize("b,hw,rw,alphabet", [(400, 39, 10, 3), (300, 80, 64, 4), (200, 59, 64, 53), (37, 300, 33, 5)])
def test_edit_distance_matches_reference(rt, b, hw, rw, alphabet):
    hyp, ref, hl, rl, exp = _edit_case(b + hw, b, hw, rw, alphabet)
    dev = lambda a: torch.from_numpy(a).to(rt.device)
    # with length arrays: the entries beyond a row's length hold symbols that must not be read
    got = ops.edit_distance(rt, dev(hyp), dev(ref), dev(hl), dev(rl))
    assert np.array_equal(got.cpu().numpy(), exp)
    # without: -1 padding ends each row
    hp, rp = hyp.copy(), ref.copy()
    for i in range(b):
        hp[i, hl[i]:], rp[i, rl[i]:] = -1, -1
    totals = torch.zeros(4, device=rt.device, dtype=torch.int64)
    for _ in range(3):
        got = ops.edit_distance(rt, dev(hp), dev(rp), totals=totals)
        assert np.array_equal(got.cpu().numpy(), exp)
    want = [3 * int(exp.sum()), 3 * int(rl.sum()), 3 * int((exp == 0).sum()), 3 * b]
    assert totals.cpu().tolist() == want


def test_edit_distance_limits(rt):
    h = torch.zeros((4, 8), device=rt.device, dtype=torch.int32)
    with pytest.raises(abi.SganError):
        ops.edit_distance(rt, h, torch.zeros((4, 65), device=rt.device, dtype=torch.int32))
    with pytest.raises(abi.SganError):
        ops.softmax_rows(rt, torch.zeros((4, 1), device=rt.device))
    with pytest.raises(abi.SganError):
        ops.ctc_greedy_decode(rt, torch.zeros((2, 30000, 3), device=rt.device))


# ----------------------------------------------------------------------------------------------------
# Recognizer.frame_probs
# ----------------------------------------------------------------------------------------------------
def _oracle_probs(x, P, mode):
    O.set_operand_rounding("bf16" if mode == "bf16" else None, wgrad=False)
    try:
        with torch.no_grad():
            return O.recognizer_probs(x, P)
    finally:
        O.set_operand_rounding(None)


def _recognizer(rt, P, classes):
    R = na.make_recognizer(IN_DIM, None, classes, vis_model=False, rt=rt, initialise=False)
    R.load_state_dict(P)
    return R


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("b,l,classes,moving", [(256, 10, 81, False), (6, 4, 53, True)])
def test_frame_probs_matches_oracle(rt, mode, b, l, classes, moving):
    rt.set_mode(mode)
    try:
        dt = torch.float64 if b < 16 else torch.float32
        P = O.make_recognizer_params(80 + b, dt, output_classes=classes, bias_scale=0.02)
        g = torch.Generator().manual_seed(81)
        if moving:                                                # inference BN: moving statistics that matter
            for k in P:
                if k.endswith("moving_mean"):
                    P[k] = torch.randn(P[k].shape, generator=g, dtype=dt) * 0.1
                if k.endswith("moving_var"):
                    P[k] = 0.5 + torch.rand(P[k].shape, generator=g, dtype=dt)
        x = torch.rand(b, 32, 16 * l, 1, generator=g, dtype=dt) * 2 - 1
        exp = _oracle_probs(x, P, mode)
        R = _recognizer(rt, P, classes)
        moving = [bn.moving_mean.data for bn in (R.bn5, R.bn6)] + [bn.moving_var.data for bn in (R.bn5, R.bn6)]
        before = [t.clone() for t in moving]
        R.bn_training = True                                      # must be ignored
        got = R.frame_probs(x.float().numpy())
        assert R.bn_training is True
        R.bn_training = False
        assert torch.equal(got, R.frame_probs(x.float().to(rt.device))), "frame_probs depends on bn_training"
        assert tuple(got.shape) == (b, 4 * l - 1, classes) and got.dtype == torch.float32 and got.is_cuda
        assert all(torch.equal(a, b) for a, b in zip(moving, before)), "frame_probs changed a moving statistic"
        err = rel_elementwise(got, exp, 1e-2) if mode == "fp32" else rel_max(got, exp)
        tol = 1e-4 if mode == "fp32" else TOL_BF16
        assert err <= tol, "{} frame_probs at B={}: rel err {:.3e} > {:.0e}".format(mode, b, err, tol)
    finally:
        rt.set_mode("fp32")


# launches of Recognizer.forward (+ its CTC) at config 3's shape, measured at the commit that introduced frame_probs: the
# trunk shared with frame_probs must not add or remove a launch of the train step
FORWARD_LAUNCHES = {"fp32": 17, "bf16": 17}


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_recognizer_forward_launches_unchanged(rt, mode):
    rt.set_mode(mode)
    try:
        R = na.make_recognizer(IN_DIM, None, 81, vis_model=False, rt=rt, seed=9)
        x = torch.rand(256, 32, 160, 1, device=rt.device) * 2 - 1
        y = torch.randint(0, 80, (256, 10), device=rt.device, dtype=torch.int32)
        R.forward(rt, x, y)
        n0 = rt.launch_count()
        R.forward(rt, x, y)
        n = rt.launch_count() - n0
        print("{} Recognizer.forward launches: {}".format(mode, n))
        assert n == FORWARD_LAUNCHES[mode], (mode, n)
    finally:
        rt.set_mode("fp32")


# ----------------------------------------------------------------------------------------------------
# public decode module
# ----------------------------------------------------------------------------------------------------
def test_ctc_decode_of_frame_probs(rt):
    rt.set_mode("fp32")
    b, l, classes = 64, 6, 53
    P = O.make_recognizer_params(90, torch.float64, output_classes=classes, bias_scale=0.3)
    g = torch.Generator().manual_seed(91)
    x = torch.rand(b, 32, 16 * l, 1, generator=g, dtype=torch.float64) * 2 - 1
    il = torch.randint(1, 4 * l, (b,), generator=g).int()
    R = _recognizer(rt, P, classes)
    probs = R.frame_probs(x.float().numpy())
    (dec,), log_prob = decode.ctc_decode(probs, il)
    assert dec.dtype == torch.int32 and tuple(dec.shape) == (b, 4 * l - 1) and tuple(log_prob.shape) == (b, 1)
    words, score = ctc_greedy_decode(probs, il.numpy())
    assert np.array_equal(dec.cpu().numpy(), _padded(words, 4 * l - 1))
    _assert_scores_close(log_prob.view(-1).cpu().numpy(), score)
    # against the fp64 oracle's own probabilities, on the samples without a near-tie among the two best classes of a frame
    exp = _oracle_probs(x, P, "fp32")
    words64, _ = ctc_greedy_decode(exp, il.numpy())
    top2 = exp.topk(2, dim=-1).values
    near = (top2[..., 0] - top2[..., 1]) < 1e-4
    checked = 0
    for i in range(b):
        if not bool(near[i, :int(il[i])].any()):
            checked += 1
            assert words[i] == words64[i], "sample {}: {} vs fp64 oracle {}".format(i, words[i], words64[i])
    assert checked >= b // 4, checked


def _scores_from(dists, ref_lens):
    d, c = int(np.sum(dists)), int(np.sum(ref_lens))
    return {"cer": d / c, "word_accuracy": float(np.mean(np.asarray(dists) == 0)), "words": len(dists), "chars": c}


def test_evaluate_recognizer(rt):
    rt.set_mode("fp32")
    classes = 53
    P = O.make_recognizer_params(95, torch.float32, output_classes=classes, bias_scale=0.3)
    R = _recognizer(rt, P, classes)
    g = torch.Generator().manual_seed(96)
    batches = []
    for b, l in ((32, 3), (16, 7)):
        batches.append((torch.rand(b, 32, 16 * l, 1, generator=g) * 2 - 1, torch.randint(0, classes - 1, (b, l), generator=g)))
    b, l = 12, 5                                                  # a ragged batch: per-sample lengths, padded labels
    lens = torch.randint(1, l + 1, (b,), generator=g)
    lens[0] = l
    labels = torch.randint(0, classes - 1, (b, l), generator=g)
    batches.append((torch.rand(b, 32, 16 * l, 1, generator=g) * 2 - 1, labels, 4 * lens - 1, lens))

    dists, ref_lens, trunk = [], [], 0
    for batch in batches:
        x = batch[0]
        n0 = rt.launch_count()
        R._logits(rt, x.to(rt.device), False)
        trunk += rt.launch_count() - n0
        probs = R.frame_probs(x)
        il = batch[2].numpy() if len(batch) > 2 else None
        words, _ = ctc_greedy_decode(probs, il)
        for i, w in enumerate(words):
            n = int(batch[3][i]) if len(batch) > 3 else batch[1].shape[1]
            ref = batch[1][i, :n].tolist()
            dists.append(levenshtein(w, ref))
            ref_lens.append(n)
    n0 = rt.launch_count()
    got = decode.evaluate_recognizer(R, iter(batches))
    launches = rt.launch_count() - n0
    assert got == _scores_from(dists, ref_lens), (got, _scores_from(dists, ref_lens))
    assert launches - trunk <= 3 * len(batches), (launches, trunk)


def test_evaluate_generated_words(rt):
    rt.set_mode("fp32")
    P = O.make_recognizer_params(97, torch.float32, output_classes=53, bias_scale=0.3)
    R = _recognizer(rt, P, 53)
    G = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, initialise=False)
    G.load_state_dict(O.make_generator_params(98, torch.float32, sigma=0.2, bias_scale=0.05))
    g = torch.Generator().manual_seed(99)
    lens = [6, 1, 3, 2, 6, 4, 5]
    labels = _padded([torch.randint(0, 52, (n,), generator=g).tolist() for n in lens], 6)
    z = torch.randn(7, 128, generator=g)
    out = decode.evaluate_generated_words(G, R, labels, noise=z)
    # the composition of the public pieces
    y = torch.from_numpy(labels).to(rt.device)
    imgs = G([z.to(rt.device), y], training=False, ragged=True)
    il = torch.tensor([4 * n - 1 for n in lens], dtype=torch.int32)
    (dec,), _ = decode.ctc_decode(R.frame_probs(imgs), il)
    dist = decode.edit_distance(dec, labels).cpu().numpy()
    assert torch.equal(out["decoded"], dec)
    assert {k: v for k, v in out.items() if k != "decoded"} == _scores_from(dist, lens)
    again = decode.evaluate_generated_words(G, R, labels, noise=z)
    assert torch.equal(again["decoded"], out["decoded"]) and {k: v for k, v in again.items() if k != "decoded"} == \
        {k: v for k, v in out.items() if k != "decoded"}
    drawn = decode.evaluate_generated_words(G, R, labels)           # z from the runtime's random stream
    assert drawn["words"] == 7 and drawn["chars"] == sum(lens)
    assert len(decode.to_strings(out["decoded"], [chr(97 + i) for i in range(52)])) == 7
