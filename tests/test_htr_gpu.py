"""Training R on its own on the GPU (scrabble-gan_b200/htr.py): the word-augmentation kernel against the float64 reference,
the HTR step against the oracle with training-mode BatchNorm (fp32, and at config-3 size in fp32 / tf32 / bf16), ragged steps, the
batch sources of generated words, determinism and state, and an end-to-end run in which R learns to read."""
import importlib

import numpy as np
import pytest
import torch
from scipy import ndimage

import _htr_ref as H
import sgan_oracle as O
from _parity import IN_DIM, _recognizer, assert_grads, grad_profile, build_models, du, make_inputs, make_params, na, nl, optim, rel_elementwise, run_step
from test_models_gpu import check_dict
from test_parity_benchpath_gpu import TOL, TOL_OUT

pytestmark = pytest.mark.gpu
ops = importlib.import_module("scrabble-gan_b200.ops")
abi = importlib.import_module("scrabble-gan_b200._abi")
htr = importlib.import_module("scrabble-gan_b200.htr")
decode = importlib.import_module("scrabble-gan_b200.decode")

AUG = dict(rotation=2.0, shear=0.3, scale=0.1, translate=2.0, p_morph=0.25)


def _smooth_words(n, w, seed):
    """Word-like test images in [-1, 1]: smoothed noise, so that the warp's fp32 coordinates (|x - c| <= 80 pixels) move a
    value by far less than the 1e-5 tolerance."""
    rng = np.random.default_rng(seed)
    img = ndimage.gaussian_filter(rng.standard_normal((n, 32, w)), sigma=(0, 2.0, 2.0), mode="nearest")
    img = img / np.abs(img).max(axis=(1, 2), keepdims=True)
    return img.astype(np.float32)


def _uniform(n, seed):
    return torch.from_numpy(np.random.default_rng(seed).uniform(-1, 1, (n, 7)).astype(np.float32))


# ----------------------------------------------------------------------------------------------------
# the augmentation kernel
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ragged", [False, True], ids=["b256_w160", "ragged_16_160"])
@pytest.mark.parametrize("ranges", ["default", "wide"])
def test_word_augment_matches_reference(rt, ragged, ranges):
    n, w = 256, 160
    kw = AUG if ranges == "default" else dict(rotation=10.0, shear=0.5, scale=0.25, translate=5.0, p_morph=0.5)
    img = _smooth_words(n, w, 1 + int(ragged))
    u = _uniform(n, 3 + int(ragged))
    widths = np.random.default_rng(5).integers(1, 11, n).astype(np.int32) * 16 if ragged else None
    x = torch.from_numpy(img).to(rt.device).view(n, 32, w, 1)
    wd = torch.from_numpy(widths).to(rt.device) if ragged else None
    got = ops.word_augment(rt, x, u.to(rt.device), wd, **kw)
    exp = H.augment(img, u.numpy(), widths, **kw)
    g = got.view(n, 32, w).cpu().numpy()
    err = np.abs(g - exp).max()
    assert err <= 1e-5, "augmentation: max abs error {:.3e} > 1e-5".format(err)
    if ragged:
        for b in range(n):
            assert np.array_equal(g[b, :, widths[b]:].view(np.int32), img[b, :, widths[b]:].view(np.int32)), b
    again = ops.word_augment(rt, x, u.to(rt.device), wd, **kw)
    assert torch.equal(again.view(torch.int32), got.view(torch.int32)), "two launches with the same u differ"


def test_word_augment_zero_ranges_copy_bits(rt):
    n, w = 64, 160
    x = torch.from_numpy(_smooth_words(n, w, 7)).to(rt.device).view(n, 32, w, 1)
    x[0, 0, 0, 0] = -0.0
    u = ops.random_(rt, rt.empty((n, 7)), normal=False)
    wd = torch.full((n,), 96, device=rt.device, dtype=torch.int32)
    for widths in (None, wd):
        got = ops.word_augment(rt, x, u, widths)
        assert torch.equal(got.view(torch.int32), x.view(torch.int32))


def test_word_augment_rejects_bad_arguments(rt):
    n, w = 4, 32
    x = rt.empty((n, 32, w, 1)).zero_()
    u = rt.empty((n, 7)).zero_()
    p = abi.ptr
    with pytest.raises(abi.SganError, match="overlaps"):
        ops.word_augment(rt, x, u, out=x)
    with pytest.raises(abi.SganError, match="32 rows"):
        ops.word_augment(rt, rt.empty((n, 16, w, 1)), u)
    with pytest.raises(abi.SganError, match="n = -1"):
        abi.call.sg_word_augment(rt.ctx, p(x), p(rt.empty(x.shape)), -1, 32, w, None, p(u), 0.0, 0.0, 0.0, 0.0, 0.0)
    with pytest.raises(abi.SganError, match="p_morph"):
        ops.word_augment(rt, x, u, p_morph=0.6)
    with pytest.raises(abi.SganError, match="scale"):
        ops.word_augment(rt, x, u, scale=1.0)
    with pytest.raises(abi.SganError, match="finite"):
        ops.word_augment(rt, x, u, rotation=-1.0)
    for bad in ([0, 16, 16, 16], [16, 16, 16, 33]):
        with pytest.raises(abi.SganError, match="widths"):
            htr.augment_words(x, bad)


# ----------------------------------------------------------------------------------------------------
# the HTR step against the oracle
# ----------------------------------------------------------------------------------------------------
def _r_params(seed, classes, dt=torch.float64, bias_scale=0.1):
    """Recogniser weights with non-trivial BatchNorm parameters, as test_recognizer_fwd_bwd uses them."""
    P = O.make_recognizer_params(seed, dt, output_classes=classes, bias_scale=bias_scale)
    g = torch.Generator().manual_seed(seed + 1)
    for k in ("bn5", "bn6"):
        P[k + ".moving_mean"] = (torch.randn(512, generator=g, dtype=torch.float64) * 0.1).to(dt)
        P[k + ".moving_var"] = (torch.rand(512, generator=g, dtype=torch.float64) + 0.5).to(dt)
        P[k + ".gamma"] = (torch.rand(512, generator=g, dtype=torch.float64) + 0.5).to(dt)
        P[k + ".beta"] = (torch.randn(512, generator=g, dtype=torch.float64) * 0.1).to(dt)
    return P


def _r_opt(lr=1e-3, beta_1=0.5, rmsprop=0):
    return optim.setup_optimizer(lr, lr, lr, lr, beta_1, 0.999, nl.hinge, 1, 0, rmsprop)[2]


def test_step_matches_oracle_fp32(rt):
    rt.set_mode("fp32")
    b, l, classes = 4, 3, 53
    P = _r_params(12, classes)
    g = torch.Generator().manual_seed(1)
    x = torch.rand(b, 32, 16 * l, 1, generator=g, dtype=torch.float64) * 2 - 1
    y = torch.randint(0, classes - 1, (b, l), generator=g)
    leaf = {k: v.clone().requires_grad_(not k.endswith(O.NON_TRAINABLE_SUFFIXES)) for k, v in P.items()}
    loss, new_stats = H.recognizer_train(x, y, torch.full((b, 1), 4 * l - 1), torch.full((b, 1), l), leaf)
    loss.sum().backward()

    R = _recognizer(rt, P, classes)
    opt = _r_opt()
    R.bn_training = False
    got = htr.train_recognizer_step(R, opt, x.float().numpy(), y.numpy().astype(np.int32))
    assert got.dim() == 0 and got.is_cuda
    assert abs(float(got) - float(loss.detach().mean())) <= 1e-4 * abs(float(loss.detach().mean()))
    assert R.bn_training is False
    grads = R.store.grad_dict()
    check_dict(grads, {k: v.grad for k, v in leaf.items() if v.grad is not None}, 1e-3, "R grads (training-mode BN)")
    sd = R.state_dict()
    for k, v in new_stats.items():
        assert float((sd[k].double().cpu() - v).abs().max() / v.abs().max()) <= 1e-4, k
    # the Keras Adam step on the gradient the step computed
    for v in R.store.trainable_variables:
        w0 = P[v.name].double()
        exp, _, _ = O.adam_update(w0, grads[v.name].double().cpu(), torch.zeros_like(w0), torch.zeros_like(w0), 1, lr=1e-3, beta1=0.5)
        assert float((sd[v.name].double().cpu() - exp).abs().max()) <= 1e-6, v.name


def _oracle_step_grads(P, x, y, l, rounding):
    leaf = {k: v.clone().requires_grad_(not k.endswith(O.NON_TRAINABLE_SUFFIXES)) for k, v in P.items()}
    b = x.shape[0]
    O.set_operand_rounding(rounding)
    try:
        loss, new_stats = H.recognizer_train(x, y, torch.full((b, 1), 4 * l - 1), torch.full((b, 1), l), leaf)
        loss.sum().backward()
    finally:
        O.set_operand_rounding(None)
    return loss.detach(), new_stats, {k: v.grad for k, v in leaf.items() if v.grad is not None}


@pytest.mark.parametrize("mode", ["fp32", "tf32", "bf16"])
def test_step_at_config3_size(rt, mode):
    """fp32 is held to TOL["fp32"].  With training-mode BatchNorm, R's gradient is far more sensitive to operand rounding than
    in inference mode: rounding the operands moves the oracle's own gradient by 1.7e-2 (tf32) and 4.9e-2 (bf16) relative L2
    at this size, against 1.1e-3 and 7.8e-3 with BN on the moving statistics (measured on the CPU oracle).  The rounding oracle
    mirrors the CUDA path's rounding points but not every rounding bit for bit, so in tf32 / bf16 the step is held to
    TOL[mode] or, where larger, to that sensitivity itself (per tensor: 5x, TOL's own ratio): the CUDA gradient must agree
    with the rounding oracle at least as well as the rounding oracle agrees with the unrounded one."""
    rt.set_mode(mode)
    try:
        b, l, classes = 256, 10, 81
        P = _r_params(70, classes, torch.float32, bias_scale=0.02)
        g = torch.Generator().manual_seed(71)
        x = torch.rand(b, 32, 16 * l, 1, generator=g) * 2 - 1
        y = torch.randint(0, classes - 1, (b, l), generator=g)
        loss, new_stats, exp = _oracle_step_grads(P, x, y, l, {"fp32": None, "tf32": "tf32", "bf16": "bf16"}[mode])
        tw, tt = TOL[mode]
        if mode != "fp32":
            sens = grad_profile(exp, _oracle_step_grads(P, x, y, l, None)[2])[0]
            tw, tt = max(tw, sens), max(tt, 5 * sens)
            print("{}: rounding moves the oracle's gradient by {:.3e}; bounds {:.2e} / {:.2e}".format(mode, sens, tw, tt))
        R = _recognizer(rt, P, classes)
        got = htr.train_recognizer_step(R, _r_opt(), x.to(rt.device), y.to(rt.device, torch.int32))
        tol_out = 1e-4 if mode == "fp32" else TOL_OUT[mode]
        assert abs(float(got) - float(loss.mean())) <= tol_out * abs(float(loss.mean()))
        assert_grads(R.store.grad_dict(), exp, tw, tt, "{} R gradients of the HTR step at config-3 size".format(mode))
        sd = R.state_dict()
        for n, v in new_stats.items():
            assert float((sd[n].double().cpu() - v.double()).abs().max() / v.double().abs().max()) <= tol_out, n
    finally:
        rt.set_mode("fp32")


def test_ragged_step(rt):
    rt.set_mode("fp32")
    classes, w = 53, 160
    lens = np.arange(1, 11, dtype=np.int32).repeat(2)
    b = len(lens)
    P = _r_params(20, classes)
    g = torch.Generator().manual_seed(21)
    x = torch.rand(b, 32, w, 1, generator=g, dtype=torch.float64) * 2 - 1
    y = np.full((b, 10), -1, np.int32)
    for i, n in enumerate(lens):
        y[i, :n] = torch.randint(0, classes - 1, (n,), generator=g).numpy()
    il, ll = 4 * lens - 1, lens
    leaf = {k: v.clone().requires_grad_(not k.endswith(O.NON_TRAINABLE_SUFFIXES)) for k, v in P.items()}
    loss, new_stats = H.recognizer_train(x, torch.from_numpy(np.maximum(y, 0)), torch.from_numpy(il), torch.from_numpy(ll), leaf)
    loss.sum().backward()
    # per-sample losses of R's training-mode forward with per-sample lengths
    R = _recognizer(rt, P, classes)
    R.bn_training = True
    per, _ = R.forward(rt, x.float().to(rt.device), torch.from_numpy(y).to(rt.device), want_grad=False,
                       input_length=torch.from_numpy(il).to(rt.device), label_length=torch.from_numpy(ll).to(rt.device))
    err = rel_elementwise(per, loss.detach(), 1.0)
    assert err <= 1e-4, "ragged per-sample losses: rel err {:.3e}".format(err)
    # the step itself
    R = _recognizer(rt, P, classes)
    got = htr.train_recognizer_step(R, _r_opt(), x.float().numpy(), y, il, ll)
    assert abs(float(got) - float(loss.detach().mean())) <= 1e-4 * abs(float(loss.detach().mean()))
    check_dict(R.store.grad_dict(), {k: v.grad for k, v in leaf.items() if v.grad is not None}, 1e-3, "ragged R grads")
    # with augmentation every word stays inside its own 16 len columns
    R = _recognizer(rt, P, classes)
    xa = x.float().numpy()
    xa[:, :, :, :] = -1.0
    got = htr.train_recognizer_step(R, _r_opt(), xa, y, il, ll, augment=AUG)
    assert np.isfinite(float(got))
    with pytest.raises(abi.SganError, match="does not fit"):
        htr.train_recognizer_step(R, _r_opt(), x.float().numpy()[:, :, :80], y, il, ll, augment=AUG)


# ----------------------------------------------------------------------------------------------------
# batch sources
# ----------------------------------------------------------------------------------------------------
def _generator(rt):
    return na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, seed=31)


def test_mixed_and_generated_batches(rt):
    rt.set_mode("bf16")
    try:
        G = _generator(rt)
        words = du.synthetic_random_words(10, [chr(65 + i) for i in range(52)], words_per_bucket=64, seed=4)
        rng = np.random.default_rng(6)
        real = [(rng.uniform(-1, 1, (4, 32, 16 * l, 1)).astype(np.float32), rng.integers(0, 52, (4, l)).astype(np.int32)) for l in (3, 7)]
        src = htr.mixed_word_batches(iter(real), G, words, 5)
        for images, labels in real:
            l = labels.shape[1]
            st = rt.rng_state().clone()
            x, y = next(src)
            assert tuple(x.shape) == (9, 32, 16 * l, 1) and tuple(y.shape) == (9, l)
            assert torch.equal(x[:4].cpu(), torch.from_numpy(images)) and np.array_equal(y[:4].cpu().numpy(), labels)
            assert all(list(r) in words[l - 1] for r in y[4:].cpu().tolist())
            rt.rng_state().copy_(st)
            z = ops.random_(rt, rt.empty((5, 128)))
            ref = G([z, y[4:].clone()], training=False, ragged=False)
            assert torch.equal(x[4:].view(torch.int32), ref.view(torch.int32)), "generated rows differ from G's own inference"
        gen = htr.generated_word_batches(G, words, 8, seed=2)
        for _ in range(6):
            x, y = next(gen)
            l = y.shape[1]
            assert tuple(x.shape) == (8, 32, 16 * l, 1)
            assert all(list(r) in words[l - 1] for r in y.cpu().tolist())
        empty = [list(b) for b in words]
        empty[2] = []
        with pytest.raises(ValueError, match="length 3"):
            next(htr.mixed_word_batches(iter(real[:1]), G, empty, 5))
        stub = type("StyleG", (), {"style": object(), "rt": rt})()
        with pytest.raises(ValueError, match="style"):
            next(htr.generated_word_batches(stub, words, 8))
    finally:
        rt.set_mode("fp32")


# ----------------------------------------------------------------------------------------------------
# determinism and state
# ----------------------------------------------------------------------------------------------------
def test_determinism_and_state(rt):
    rt.set_mode("bf16")
    try:
        b, l, classes = 32, 4, 53
        P = _r_params(40, classes, torch.float32, bias_scale=0.02)
        rng = np.random.default_rng(41)
        x = rng.uniform(-1, 1, (b, 32, 16 * l, 1)).astype(np.float32)
        y = rng.integers(0, classes - 1, (b, l)).astype(np.int32)
        outs = []
        for _ in range(2):
            R = _recognizer(rt, P, classes)
            opt = _r_opt()
            rt.manual_seed(99)
            for _ in range(2):
                htr.train_recognizer_step(R, opt, x, y, augment=AUG)
            outs.append((R.store.w.clone(), R.state_dict()))
        assert torch.equal(outs[0][0], outs[1][0]), "weights differ between two identical runs"
        for k in ("bn5.moving_mean", "bn5.moving_var", "bn6.moving_mean", "bn6.moving_var"):
            assert torch.equal(outs[0][1][k], outs[1][1][k]), k

        class Boom:
            def apply_gradients(self, gv):
                raise RuntimeError("boom")
        for flag in (False, True):
            R.bn_training = flag
            with pytest.raises(RuntimeError, match="boom"):
                htr.train_recognizer_step(R, Boom(), x, y)
            assert R.bn_training is flag
        R.bn_training = False

        # a GAN step still runs afterwards, on a recogniser trained on its own
        Pg = make_params(42, torch.float32, r_classes=53)
        G, D, R2, _ = build_models(rt, Pg)
        images, labels, fake, z = make_inputs(43, 2, 2, 2, torch.float32)
        htr.train_recognizer_step(R2, _r_opt(), images.numpy(), labels.numpy().astype(np.int32))
        stats, _ = run_step(rt, G, D, R2, None, images, labels, fake, z)
        assert all(np.isfinite(v) for v in stats.values()), stats
    finally:
        rt.set_mode("fp32")


# ----------------------------------------------------------------------------------------------------
# R learns to read
# ----------------------------------------------------------------------------------------------------
N_CLASSES = 20                 # letters; R has one more output (the blank)
# (steps, Adam learning rate): the second, slower phase lets BatchNorm's moving statistics (momentum 0.99), which
# evaluate_recognizer reads with, catch up with weights that stop moving fast
LEARN_PHASES = ((400, 1e-3), (300, 1e-4))


def _glyphs(seed):
    """Per-class 32x16 glyphs: a random 6x3 block pattern (ink +1 on background -1) inside a 2-pixel background border."""
    rng = np.random.default_rng(seed)
    out = np.full((N_CLASSES, 32, 16), -1.0, np.float32)
    for c in range(N_CLASSES):
        pat = rng.random((6, 3)) < 0.45
        out[c, 4:28, 2:14] = np.where(np.kron(pat, np.ones((4, 4))) > 0, 1.0, -1.0)
    return out


def _word_batches(glyphs, batch, seed):
    rng = np.random.default_rng(seed)
    while True:
        l = int(rng.integers(1, 6))
        y = rng.integers(0, N_CLASSES, (batch, l)).astype(np.int32)
        x = np.concatenate([glyphs[y[:, i]] for i in range(l)], axis=2) + rng.normal(0, 0.2, (batch, 32, 16 * l)).astype(np.float32)
        yield np.clip(x, -1, 1)[..., None].astype(np.float32), y


def test_recognizer_learns_to_read(rt):
    rt.set_mode("bf16")
    try:
        glyphs = _glyphs(50)
        R = na.make_recognizer(IN_DIM, None, N_CLASSES + 1, vis_model=False, rt=rt, seed=51)
        opt = optim.setup_optimizer(1e-3, 1e-3, 1e-3, 1e-3, 0.9, 0.999, nl.hinge, 1, 0, 0)[2]
        train = _word_batches(glyphs, 64, 52)
        held = [next(_word_batches(glyphs, 64, 53 + i)) for i in range(8)]
        losses = []
        for steps, lr in LEARN_PHASES:
            opt.learning_rate = lr
            for _ in range(steps):
                losses.append(htr.train_recognizer_step(R, opt, *next(train), augment=AUG))
            scores = decode.evaluate_recognizer(R, held)
            print("R learns: after {} steps (lr {:.0e}) held-out CER {:.4f}, word accuracy {:.4f}".format(
                len(losses), lr, scores["cer"], scores["word_accuracy"]))
        losses = torch.stack(losses).cpu().numpy()
        print("R learns: loss {:.3f} -> {:.3f} (mean of the last 10 steps)".format(losses[0], losses[-10:].mean()))
        assert scores["words"] == 512
        assert scores["cer"] < 0.05, scores
        assert losses[-10:].mean() < 0.1 * losses[0], (losses[0], losses[-10:])
    finally:
        rt.set_mode("fp32")
