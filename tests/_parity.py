"""Shared helpers of the GPU parity tests: error metrics that CAN fail, and failure messages that carry the whole
per-tensor table (a GPU run is expensive: one failing run must say everything)."""
import importlib

import numpy as np
import torch

import sgan_oracle as O

na = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture")
du = importlib.import_module("scrabble-gan_b200.bigacgan.data_utils")
nl = importlib.import_module("scrabble-gan_b200.bigacgan.net_loss")
optim = importlib.import_module("scrabble-gan_b200.optim")

IN_DIM = (32, 160, 1)


def _flat(t):
    return torch.as_tensor(t).detach().double().cpu().reshape(-1)


def grad_profile(got, exp, skip=()):
    """Relative L2 error of the WHOLE gradient of one network (all tensors concatenated) and of every tensor.  A tensor's
    error is taken relative to max(its own norm, 1e-3 x the whole gradient's norm): tensors whose true gradient is
    (analytically or numerically) negligible -- e.g. the bias of a transposed conv that feeds a batch-norm -- are judged
    against that floor instead of against their own round-off."""
    num = den = 0.0
    rows = []
    for k, e in exp.items():
        if k in skip or k.endswith(O.NON_TRAINABLE_SUFFIXES):
            continue
        g, e = _flat(got[k]), _flat(e)
        assert g.shape == e.shape, (k, g.shape, e.shape)
        assert torch.isfinite(g).all(), "non-finite gradient in " + k
        d2, e2 = float(((g - e) ** 2).sum()), float((e ** 2).sum())
        num, den = num + d2, den + e2
        rows.append([k, d2, e2])
    floor2 = 1e-6 * den
    per = {k: (d2 / max(e2, floor2, 1e-300)) ** 0.5 for k, d2, e2 in rows}
    share = {k: (e2 / max(den, 1e-300)) ** 0.5 for k, d2, e2 in rows}
    return (num / max(den, 1e-300)) ** 0.5, per, share


class Soft:
    """Collects failed checks so that ONE (expensive) GPU run reports everything that is off, then fails at the end."""

    def __init__(self):
        self.msgs = []

    def check(self, cond, msg):
        print(("ok   " if cond else "FAIL ") + msg.split("\n")[0])
        if not cond:
            self.msgs.append(msg)

    def done(self):
        assert not self.msgs, "\n".join(self.msgs)


def assert_grads(got, exp, tol_whole, tol_tensor, what, skip=(), soft=None):
    """whole-gradient rel L2 <= tol_whole AND every tensor's rel L2 (see grad_profile) <= tol_tensor."""
    whole, per, share = grad_profile(got, exp, skip)
    worst = sorted(per.items(), key=lambda kv: -kv[1])
    table = "\n".join("    {:<28s} err {:.3e}   norm share {:.3e}".format(k, v, share[k]) for k, v in worst[:12])
    msg = "{}: whole-gradient rel L2 {:.3e} (bound {:.1e}); worst tensors (bound {:.1e}):\n{}".format(what, whole, tol_whole, tol_tensor, table)
    ok = whole <= tol_whole and worst[0][1] <= tol_tensor
    if soft is not None:
        soft.check(ok, msg)
    else:
        print(msg)
        assert ok, msg
    return whole, worst[0]


def rel_max(got, exp, floor=1e-5):
    """max |got - exp| / max |exp|."""
    g, e = _flat(got), _flat(exp)
    assert g.shape == e.shape, (g.shape, e.shape)
    assert torch.isfinite(g).all(), "non-finite values"
    return float((g - e).abs().max() / max(float(e.abs().max()), floor))


def rel_elementwise(got, exp, floor_frac=1e-2):
    """max over elements of |got - exp| / max(|exp|, floor_frac * max|exp|): an ELEMENTWISE relative error (entries that are
    small next to the tensor's scale are judged against floor_frac of that scale)."""
    g, e = _flat(got), _flat(exp)
    assert g.shape == e.shape, (g.shape, e.shape)
    assert torch.isfinite(g).all(), "non-finite values"
    den = torch.clamp(e.abs(), min=floor_frac * float(e.abs().max()))
    return float(((g - e).abs() / den).max())


def assert_stats(got, exp, tol, what, floor=1e-2, soft=None, tol_by_name=None):
    bad = []
    for k in O.STAT_NAMES:
        e, g = float(exp[k]), float(got[k])
        err = abs(g - e) / max(abs(e), floor)
        if not np.isfinite(g) or err > (tol_by_name or {}).get(k, tol):
            bad.append("{}: got {!r} expected {!r} (rel {:.2e})".format(k, g, e, err))
    msg = "{} statistics beyond {:.0e}:\n  ".format(what, tol) + "\n  ".join(bad)
    if soft is not None:
        soft.check(not bad, msg if bad else "{} statistics within {:.0e}".format(what, tol))
    else:
        assert not bad, msg


def make_params(seed, dt, sigma=0.2, bias_scale=0.05, use_w=False, style_encoder=False, r_classes=53):
    P = {"G": O.make_generator_params(seed + 1, dt, sigma=sigma, bias_scale=bias_scale, style_encoder_too=style_encoder),
         "D": O.make_discriminator_params(seed + 2, dt, sigma=sigma, bias_scale=bias_scale),
         "R": O.make_recognizer_params(seed + 3, dt, output_classes=r_classes, bias_scale=bias_scale)}
    if use_w:
        P["W"] = O.make_discriminator_params(seed + 4, dt, sigma=sigma, bias_scale=bias_scale)
    return P


def make_inputs(seed, b, l_r, l_f, dt):
    g = torch.Generator().manual_seed(seed)
    images = torch.rand(b, 32, 16 * l_r, 1, generator=g, dtype=dt) * 2 - 1
    labels = torch.randint(0, 52, (b, l_r), generator=g)
    fake_labels = torch.randint(0, 52, (b, l_f), generator=g)
    z = torch.randn(b, 128, generator=g, dtype=dt)
    return images, labels, fake_labels, z


def build_models(rt, P, style_encoder=False, r_classes=53):
    """libsgan models carrying the oracle's weights (initialise=False: construction launches nothing but copies)."""
    G = na.make_generator(128, IN_DIM, (32, 8192), None, "B3", 52, vis_model=False, rt=rt, style_encoder=style_encoder, initialise=False)
    D = na.make_discriminator(IN_DIM, None, "B1", vis_model=False, rt=rt, initialise=False)
    R = na.make_recognizer(IN_DIM, None, r_classes, vis_model=False, rt=rt, initialise=False)
    G.load_state_dict(P["G"]); D.load_state_dict(P["D"]); R.load_state_dict(P["R"])
    W = None
    if "W" in P:
        W = na.make_style_promoter(IN_DIM, None, "B1", vis_model=False, rt=rt, initialise=False)
        W.load_state_dict(P["W"])
    return G, D, R, W


def _recognizer(rt, P, classes):
    """A libsgan recogniser of `classes` outputs carrying the weights P."""
    R = na.make_recognizer(IN_DIM, None, classes, vis_model=False, rt=rt, initialise=False)
    R.load_state_dict(P)
    return R


def run_step(rt, G, D, R, W, images, labels, fake_labels, z, loss_name="hinge", balance=True, style=None, batch_idx=0):
    gan = na.make_gan(G, D, R, W, vis_model=False)
    g_opt, d_opt, r_opt, w_opt, loss_fn, disc_iters, agb = optim.setup_optimizer(2e-4, 2e-4, 2e-4, 2e-4, 0.0, 0.999, getattr(nl, loss_name), 1,
                                                                                 int(balance), 0)
    b = images.shape[0]
    out = du.train_step(0, batch_idx, 1, images.float().numpy(), labels.numpy(), D, R, W, gan, g_opt, d_opt, r_opt, w_opt,
                        [s.numpy() for s in style.float()] if style is not None else None, b, 128, loss_fn, disc_iters, agb,
                        None, 10, "", fake_labels=fake_labels.numpy(), noise=None if G.style is not None else z.float().numpy())
    assert len(out) == 16
    return dict(zip(du.STAT_NAMES, out)), (g_opt, d_opt, r_opt, w_opt)
