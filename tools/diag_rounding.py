"""GPU diagnostic: where do the reduced-precision modes of the CUDA path differ from the oracle's operand-rounding model?
(1) how the tensor core reads fp32 as tf32 (truncate / round-to-nearest), (2) per-network isolation in bf16 / tf32 mode
(D, R, G forward + backward against the rounded oracle, attention on and off).  Run under gpurun; prints tables."""
import importlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import torch  # noqa: E402

import sgan_oracle as O  # noqa: E402
from _parity import build_models, grad_profile, make_params, rel_max  # noqa: E402

runtime = importlib.import_module("scrabble-gan_b200.runtime")
ops = importlib.import_module("scrabble-gan_b200.ops")
abi = importlib.import_module("scrabble-gan_b200._abi")
F32, BF16 = abi.SG_F32, abi.SG_BF16


def table(title, got, exp):
    whole, per, share = grad_profile(got, exp)
    print("  {}: whole {:.3e}".format(title, whole))
    for k, v in sorted(per.items(), key=lambda kv: -kv[1])[:8]:
        print("      {:<26s} {:.3e}  share {:.2e}".format(k, v, share[k]))


def tf32_mode_probe(rt):
    rt.set_mode("tf32")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 8, 8, 64, generator=g)
    w = torch.randn(3, 3, 64, 64, generator=g) * 0.1
    d = ops.desc_conv_fwd(2, 8, 8, 64, 64, 3, 3, "same", F32, F32)
    xd, wd = x.to(rt.device), w.to(rt.device)
    packed = ops.pack_weights(rt, d, wd)
    out = torch.empty(2, 8, 8, 64, device=rt.device)
    ops.conv_run(rt, d, xd, wd, packed, None, None, out)
    rt.sync()

    def rn(t):
        i = t.float().contiguous().view(torch.int32)
        i = ((i + 0x0FFF + ((i >> 13) & 1)) & ~0x1FFF)
        return i.view(torch.float32).double()

    def rna(t):      # round half away from zero on the magnitude
        i = t.float().contiguous().view(torch.int32)
        i = ((i + 0x1000) & ~0x1FFF)
        return i.view(torch.float32).double()

    def tr(t):
        return O._q_tf32(t).double()
    for name, f in (("truncate", tr), ("round-nearest-even", rn), ("round-half-away", rna), ("exact fp32 operands", lambda t: t.double())):
        ref = O.conv2d(f(x), f(w))
        print("  tf32 conv vs {:<22s}: rel max err {:.3e}".format(name, rel_max(out, ref)))


def d_isolation(rt, mode, sigma):
    rt.set_mode(mode)
    dt = torch.float64
    P = make_params(40, dt, sigma=sigma)
    g = torch.Generator().manual_seed(5)
    b, l = 4, 3
    x = (torch.rand(b, 32, 16 * l, 1, generator=g, dtype=dt) * 2 - 1).requires_grad_(True)
    up = torch.randn(b, generator=g, dtype=dt)
    O.set_operand_rounding(mode if mode != "fp32" else None, wgrad=(mode == "bf16"))
    try:
        leaf = {k: v.clone().requires_grad_(True) for k, v in P["D"].items()}
        # per-block activations
        acts = []
        net = x
        for i in range(4):
            net = O.resnet_block_down(net, leaf, "B%d" % (i + 1), i == 3)
            if i == 0:
                net = O.non_local_block(net, leaf, "B1.attn")
            acts.append(net.detach())
        logits = O.discriminator(x, leaf, "B1")
        (logits.view(-1) * up).sum().backward()
    finally:
        O.set_operand_rounding(None)
    _, D, _, _ = build_models(rt, P)
    D.store.zero_grad()
    xd = x.detach().float().to(rt.device)
    net = xd
    print("D isolation mode={} sigma={}".format(mode, sigma))
    for i, blk in enumerate(D.trunk.blocks):
        net, _ = blk.forward(rt, net)
        if i in D.trunk.attn:
            net, _ = D.trunk.attn[i].forward(rt, net)
        print("  after B{}: rel max err {:.3e}".format(i + 1, rel_max(net, acts[i])))
    got, cache = D.forward(rt, xd)
    print("  logits: got {} exp {}".format([round(float(v), 5) for v in got.view(-1)], [round(float(v), 5) for v in logits.view(-1)]))
    dx = D.backward(rt, cache, up.float().to(rt.device), wgrad=True, want_dx=True)
    print("  d/d image: rel max err {:.3e}".format(rel_max(dx, x.grad)))
    table("D grads", D.store.grad_dict(), {k: v.grad for k, v in leaf.items()})


def r_isolation(rt, mode):
    rt.set_mode(mode)
    dt = torch.float64
    P = make_params(40, dt)
    g = torch.Generator().manual_seed(6)
    b, l = 4, 3
    x = (torch.rand(b, 32, 16 * l, 1, generator=g, dtype=dt) * 2 - 1).requires_grad_(True)
    y = torch.randint(0, 52, (b, l), generator=g)
    O.set_operand_rounding(mode if mode != "fp32" else None, wgrad=(mode == "bf16"))
    try:
        leaf = {k: v.clone().requires_grad_(not k.endswith(O.NON_TRAINABLE_SUFFIXES)) for k, v in P["R"].items()}
        loss = O.recognizer(x, y, torch.full((b, 1), 4 * l - 1), torch.full((b, 1), l), leaf)
        loss.sum().backward()
    finally:
        O.set_operand_rounding(None)
    _, _, R, _ = build_models(rt, P)
    R.store.zero_grad()
    got, cache = R.forward(rt, x.detach().float().to(rt.device), y.to(rt.device, torch.int32))
    dx = R.backward(rt, cache, None, wgrad=True, want_dx=True)
    print("R isolation mode={}: loss rel max err {:.3e}; d/d image {:.3e}".format(mode, rel_max(got, loss.view(-1)), rel_max(dx, x.grad)))
    table("R grads", R.store.grad_dict(), {k: v.grad for k, v in leaf.items() if v.grad is not None})


def g_isolation(rt, mode, sigma):
    rt.set_mode(mode)
    dt = torch.float64
    P = make_params(40, dt, sigma=sigma)
    g = torch.Generator().manual_seed(7)
    b, l = 4, 3
    z = torch.randn(b, 128, generator=g, dtype=dt)
    y = torch.randint(0, 52, (b, l), generator=g)
    O.set_operand_rounding(mode if mode != "fp32" else None, wgrad=(mode == "bf16"))
    try:
        leaf = {k: (v.clone().requires_grad_(True) if not k.endswith(O.NON_TRAINABLE_SUFFIXES) else v.clone()) for k, v in P["G"].items()}
        img = O.generator_core(z, y, leaf, "B3", True, {})
        dimg = torch.randn(img.shape, generator=g, dtype=dt)
        (img * dimg).sum().backward()
    finally:
        O.set_operand_rounding(None)
    G, _, _, _ = build_models(rt, P)
    G.store.zero_grad()
    got, cache = G.forward(rt, z.float().to(rt.device), y.to(rt.device, torch.int32), training=True)
    print("G isolation mode={} sigma={}: image rel max err {:.3e}".format(mode, sigma, rel_max(got, img)))
    G.backward(rt, cache, dimg.float().to(rt.device))
    table("G grads", G.store.grad_dict(), {k: v.grad for k, v in leaf.items() if v.requires_grad})


def cbn_gb(rt, cbn, z):
    """(gamma, beta, row stride) of one conditional BN layer from its own Dense layers; z: a block's slice of the latent."""
    return cbn.gamma.forward(rt, z, z.shape[0], ldx=128), cbn.beta.forward(rt, z, z.shape[0], ldx=128), None


def g_stages(rt, mode, sigma=0.0):
    """stage-by-stage forward of G against the (rounded) oracle"""
    rt.set_mode(mode)
    layers = importlib.import_module("scrabble-gan_b200.layers")
    dt = torch.float64
    P = make_params(40, dt, sigma=sigma)["G"]
    g = torch.Generator().manual_seed(7)
    b, l = 4, 3
    z = torch.randn(b, 128, generator=g, dtype=dt)
    y = torch.randint(0, 52, (b, l), generator=g)
    O.set_operand_rounding(mode if mode != "fp32" else None)
    try:
        zs = torch.split(z, 32, dim=1)
        exp = {}
        net = O.filter_bank(zs[0], y, P["filter_bank"])
        exp["bank"] = net
        for i in range(3):
            name = "B%d" % (i + 1)
            net = O.resnet_block_up(net, zs[i + 1], P, name, i == 2, True, {})
            exp[name] = net
            if name == "B3":
                net = O.non_local_block(net, P, name + ".attn")
                exp["attn"] = net
        xh, _, _ = O.batchnorm_train(net, P["bn.moving_mean"], P["bn.moving_var"])
        act = torch.relu(xh * P["bn.gamma"] + P["bn.beta"])
        exp["act"] = act
        exp["pre"] = O.conv2d(act, P["out.w"], P["out.b"])
    finally:
        O.set_operand_rounding(None)
    G, _, _, _ = build_models(rt, make_params(40, dt, sigma=sigma))
    zd, yd = z.float().to(rt.device), y.to(rt.device, torch.int32)
    print("G stages mode={} sigma={}".format(mode, sigma))
    net, _ = G.embed.forward(rt, zd, 128, yd)
    print("  bank : {:.3e}".format(rel_max(net, exp["bank"])))
    for i, blk in enumerate(G.blocks):
        zi = zd[:, 32 * (i + 1):]
        net, _ = blk.forward(rt, net, True, cbn_gb(rt, blk.cbn1, zi), cbn_gb(rt, blk.cbn2, zi))
        print("  B{}   : {:.3e}".format(i + 1, rel_max(net, exp["B%d" % (i + 1)])))
        if i in G.attn:
            net, _ = G.attn[i].forward(rt, net)
            print("  attn : {:.3e}".format(rel_max(net, exp["attn"])))
    mean, rstd, count = layers.batch_stats(rt, net, G.bn, update_moving=False)
    act = ops.bn_apply(rt, net, mean, rstd, G.bn.gamma.data, G.bn.beta.data, False, True, rt.op_dt)
    print("  act  : {:.3e}".format(rel_max(act.float(), exp["act"])))
    pre = G.out.forward(rt, act)
    print("  pre  : {:.3e}  (max |pre| {:.3f})".format(rel_max(pre, exp["pre"]), float(exp["pre"].abs().max())))
    # block 1 in detail
    blk = G.blocks[0]
    x0, _ = G.embed.forward(rt, zd, 128, yd)
    O.set_operand_rounding(mode if mode != "fp32" else None)
    try:
        e_a1 = torch.relu(O.conditional_batchnorm(exp["bank"], zs[1], P, "B1.cbn1", True, {}))
        e_u = O.conv2d_transpose(e_a1, P["B1.up.w"], P["B1.up.b"], (2, 2))
        e_a2 = torch.relu(O.conditional_batchnorm(e_u, zs[1], P, "B1.cbn2", True, {}))
        e_h = O.conv2d(e_a2, P["B1.conv.w"], P["B1.conv.b"])
        e_s = O.conv2d_transpose(exp["bank"], P["B1.short.w"], P["B1.short.b"], (2, 2))
    finally:
        O.set_operand_rounding(None)
    zi = zd[:, 32:]
    a1, _ = blk.cbn1.forward(rt, x0, cbn_gb(rt, blk.cbn1, zi), True, True, rt.op_dt)
    print("  B1.a1: {:.3e}".format(rel_max(a1.float(), e_a1)))
    u = blk.up.forward(rt, a1)
    print("  B1.u : {:.3e}".format(rel_max(u, e_u)))
    a2, _ = blk.cbn2.forward(rt, u, cbn_gb(rt, blk.cbn2, zi), True, True, rt.op_dt)
    print("  B1.a2: {:.3e}".format(rel_max(a2.float(), e_a2)))
    h = blk.conv.forward(rt, a2)
    print("  B1.h : {:.3e}".format(rel_max(h, e_h)))
    xs = ops.cast(rt, x0, rt.op_dt)
    sh = blk.short.forward(rt, xs, out=torch.zeros_like(h), accumulate=True)
    print("  B1.sh: {:.3e}".format(rel_max(sh, e_s)))


def main():
    rt = runtime.Runtime(device=0, mode="fp32")
    runtime.set_runtime(rt)
    if len(sys.argv) > 1 and sys.argv[1] == "g":
        for mode in ("fp32", "bf16", "tf32"):
            g_stages(rt, mode)
        return
    tf32_mode_probe(rt)
    for mode in ("bf16", "tf32"):
        for sigma in (0.0, 0.2):
            d_isolation(rt, mode, sigma)
        r_isolation(rt, mode)
        for sigma in (0.0, 0.2):
            g_isolation(rt, mode, sigma)


if __name__ == "__main__":
    main()
