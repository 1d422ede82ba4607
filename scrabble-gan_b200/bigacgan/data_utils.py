"""train_step / apply_gradient_balancing / train shell with the reference's signatures
(src/bigacgan/data_utils.py: train :198-352, train_step :358-473, apply_gradient_balancing :476-490,
generate_and_save_images :493-519).

train_step does what the reference's four GradientTapes + four apply_gradients do, as explicit forward and backward
passes over libsgan kernels:
    forward   G(z|style, fake labels);  D(fake), R(fake) [, W(fake)];  D(real) [, W(style), W(real)];  R(real)
    losses    hinge | not_saturating, gradient balancing (loss-level, differentiable std; SURVEY Q6), 16 statistics
    backward  D: d_loss -> D (real + fake branches, dgrad + wgrad);  R: r_real -> R;  W: s_loss -> W;
              G: g_final -> image through the frozen D, R (, W) (dgrad only) -> G (dgrad + wgrad)
    update    Adam x4 (one fused launch per network); gradients are of SUMS over the batch (SURVEY Q7)
Under data parallelism (runtime.world_size > 1) BN statistics, the loss sums and the gradient buckets are
sum-all-reduced over NCCL so that N replicas on shards equal one replica on the concatenated batch."""
from __future__ import annotations

import os
import random
import time

import numpy as np
import torch

from .. import ops
from .._abi import SG_LOSS_NSUMS, call
from ..ops import _p
from ..runtime import Runtime, get_runtime
from . import net_loss
from .net_architecture import _as_tensor, _nhwc, to_device_f32, to_device_i32

STAT_NAMES = ("r_loss_fake", "r_loss_real", "r_loss_balanced", "g_loss", "g_loss_added", "g_loss_balanced", "d_loss",
              "d_loss_real", "d_loss_fake", "g_loss_final", "alpha", "r_loss_fake_std", "g_loss_std", "s_loss", "s_loss_real",
              "s_loss_fake")


def apply_gradient_balancing(r_fake_logits, g_loss, alpha=1):
    """Reference data_utils.py:476-490: returns (g_balanced, r_loss_balanced, alpha, std(r_fake), std(g_loss));
    population std, no zero guard.  Inputs are (B,1) device tensors (or DLPack producers)."""
    from .._abi import from_dlpack
    rt = get_runtime()
    r = from_dlpack(r_fake_logits).to(device=rt.device, dtype=torch.float32).reshape(-1).contiguous()
    g = from_dlpack(g_loss).to(device=rt.device, dtype=torch.float32).reshape(-1).contiguous()
    b = r.numel()
    g_bal, r_bal, stds = rt.empty((b,)), rt.empty((b,)), rt.empty((2,))
    call.sg_grad_balance(rt.ctx, _p(r), _p(g), b, float(alpha), _p(g_bal), _p(r_bal), _p(stds))
    return g_bal.view(b, 1), r_bal.view(b, 1), alpha, stds[0], stds[1]


def _loss_kind(loss_fn) -> int:
    kind = getattr(loss_fn, "sg_kind", None)
    if kind is None:
        name = getattr(loss_fn, "__name__", str(loss_fn))
        if name in ("hinge", "not_saturating"):
            return getattr(net_loss, name).sg_kind
        raise ValueError("loss_fn must be net_loss.hinge or net_loss.not_saturating (got {!r})".format(loss_fn))
    return kind


# ----------------------------------------------------------------------------------------------------
# CUDA-graph replay of the step
# ----------------------------------------------------------------------------------------------------
# A step is ~390 kernel launches issued from Python through ctypes.  Once a (models, shapes, mode) signature has been
# seen GRAPH_WARMUP times, the device part of the step (everything between the input copies and the 16 statistics) is
# captured ONCE into a CUDA graph -- torch is used only as the capture / allocator plumbing -- and later calls replay it:
# inputs are copied into static device buffers, the Adam step sizes travel through pinned host scalars that captured
# memcpy nodes re-read on every replay, and the result is the same `stats` tensor.  Set SGAN_CUDA_GRAPH=0 to disable.
# "reference" = this fork's loss-level balancing (data_utils.py:476-490, the default and the parity target); "paper" = the
# gradient-level balancing of the ScrabbleGAN paper / BASELINE north_star, std(grad_D)/std(grad_R) on the image gradients
BALANCE_MODE = os.environ.get("SGAN_BALANCE_MODE", "reference")
GRAPH_ENABLED = os.environ.get("SGAN_CUDA_GRAPH", "1") != "0"
GRAPH_DP = os.environ.get("SGAN_CUDA_GRAPH_DP", "1") != "0"      # capture the data-parallel step too (NCCL + peer exchanges)
GRAPH_WARMUP = int(os.environ.get("SGAN_CUDA_GRAPH_WARMUP", "2"))   # eager calls of a signature before it is captured
# One graph per (models, B, L_real, L_fake, mode, ...) signature -- up to 100 (L_real, L_fake) pairs in training on words of
# 1..10 characters.  All graphs allocate from ONE shared memory pool (they replay one after the other on one stream, so the
# activations of one graph may reuse the memory of another): the footprint is the largest signature's, not the sum.
GRAPH_MAX = int(os.environ.get("SGAN_CUDA_GRAPH_MAX", "256"))
_graph_cache = {}
_graph_pool = [None]


class _GraphedStep:
    def __init__(self):
        self.calls = 0
        self.graph = None
        self.static = None          # (x_real, y_real, y_fake, g_in) static device buffers
        self.stats = None
        self.versions = None
        self.failed = False
        self.launches = 0           # libsgan kernel nodes in the graph
        self.owners = None          # strong references to the models / optimizers the key's id()s stand for: an id can
                                    # only be recycled after the object dies, and the graph's kernels point at its buffers


def _graph_key(rt, generator, discriminator, recognizer, opts, b, l_r, l_f, kind, balance, update_g, balance_mode="reference"):
    return (id(generator), id(discriminator), id(recognizer), tuple(id(o) for o in opts), b, l_r, l_f, rt.mode, kind, bool(balance),
            bool(update_g), bool(recognizer.trainable), balance_mode,
            tuple(bool(getattr(m, "apply_sn", False)) for m in (generator, discriminator)))


def train_step(epoch_idx, batch_idx, batch_per_epoch, images, labels, discriminator, recognizer, style_promoter, composite_gan,
               generator_optimizer, discriminator_optimizer, recognizer_optimizer, stylepromoter_optimizer, my_imgs, batch_size,
               latent_dim, loss_fn, disc_iters, apply_gradient_balance, random_words, bucket_size, gen_path, *,
               fake_labels=None, noise=None, verbose: bool = False, return_device_stats: bool = False, balance_mode: str = None):
    """One G + D + R (+ W) training step.  Positional signature = the reference's (data_utils.py:358-360); returns the
    same 16-tuple of Python floats in the same order (:470-473).

    images (B,32,16*L_r[,1]) and labels (B,L_r) may be host numpy arrays (copied H2D here), torch tensors or DLPack
    producers.  `style_promoter` may be None (G+D+R mode).  Keyword extensions: `fake_labels` (B,L_f) int and `noise`
    (B,latent_dim) make the step deterministic (the reference samples both internally; SURVEY K21); `balance_mode`
    "reference" (default: loss-level balancing, data_utils.py:476-490) or "paper" (gradient-level balancing on the image
    gradients, std(grad_D)/std(grad_R): arXiv 2003.10557 section 3.4)."""
    generator = composite_gan.generator
    balance_mode = balance_mode or BALANCE_MODE
    if balance_mode not in ("reference", "paper"):
        raise ValueError("balance_mode must be 'reference' or 'paper'")
    rt: Runtime = generator.rt
    use_w = style_promoter is not None
    kind = _loss_kind(loss_fn)

    # ---- inputs (data_utils.py:385-395) ---------------------------------------------------------------------------
    if fake_labels is None:
        random_bucket_idx = random.randint(0, bucket_size - 1)
        fake_labels = np.array([random.choice(random_words[random_bucket_idx]) for _ in range(batch_size)], np.int32)
    b, l_r = int(np.shape(labels)[0]), int(np.shape(labels)[1])
    l_f = int(np.shape(fake_labels)[1])
    update_g = (batch_idx + 1) % disc_iters == 0
    opts = (generator_optimizer, discriminator_optimizer, recognizer_optimizer, stylepromoter_optimizer)
    args = (discriminator, recognizer, style_promoter, generator, opts, kind, apply_gradient_balance, update_g, balance_mode)

    # ---- CUDA-graph path (G+D+R mode on one replica) ---------------------------------------------------------------
    graphable = (GRAPH_ENABLED and not use_w and generator.style is None and (rt.world_size == 1 or GRAPH_DP) and
                 all(type(o).__name__ == "Adam" for o in opts[:3]))
    if graphable:
        key = _graph_key(rt, generator, discriminator, recognizer, opts, b, l_r, l_f, kind, apply_gradient_balance, update_g, balance_mode)
        gs = _graph_cache.get(key)
        if gs is None:
            gs = _graph_cache[key] = _GraphedStep()
        gs.calls += 1
        if gs.graph is None and not gs.failed and gs.calls > GRAPH_WARMUP and \
                sum(1 for g_ in _graph_cache.values() if g_.graph is not None) < GRAPH_MAX:
            _capture(rt, gs, args, b, l_r, l_f, latent_dim)
        if gs.graph is not None:
            stats = _replay(rt, gs, args, images, labels, fake_labels, noise)
            return _finish(stats, return_device_stats, verbose, epoch_idx, batch_idx, batch_per_epoch)

    y_real = to_device_i32(rt, labels)
    y_fake = to_device_i32(rt, fake_labels)
    x_real = _nhwc(to_device_f32(rt, images)).reshape(b, 32, 16 * l_r, 1)
    style_imgs = None
    if generator.style is not None or use_w:
        style_imgs = _nhwc(to_device_f32(rt, my_imgs))
    if generator.style is not None:
        g_in = style_imgs
    else:
        # noise = tf.random.normal([batch_size, latent_dim]) (data_utils.py:385): libsgan's Philox kernel, no torch op
        g_in = to_device_f32(rt, noise) if noise is not None else ops.random_(rt, rt.empty((batch_size, latent_dim)))
    stats = _step_device(rt, args, x_real, y_real, y_fake, g_in, style_imgs)
    return _finish(stats, return_device_stats, verbose, epoch_idx, batch_idx, batch_per_epoch)


def _finish(stats, return_device_stats, verbose, epoch_idx, batch_idx, batch_per_epoch):
    if return_device_stats:
        return stats
    host = stats.cpu().tolist()          # the reference's 16 .numpy() calls: one D2H copy + sync here
    if verbose:
        print('>%d, %d/%d, d=%.3f, d_real=%.3f, d_fake=%.3f, g_trad=%.3f, r_loss_fake=%.3f, g_loss=%.3f, r=%.3f, s=%.3f' % (
            epoch_idx + 1, batch_idx + 1, batch_per_epoch, host[6], host[7], host[8], host[3], host[0], host[9], host[1], host[14]))
    return tuple(host)


def _capture(rt, gs, args, b, l_r, l_f, latent_dim):
    """Capture the device part of the step for this signature.  Kernels do not run during capture; Python-side state the
    body advances (optimizer iteration counters, store versions) is rolled back afterwards and advanced by _replay."""
    discriminator, recognizer, style_promoter, generator, opts, kind, balance, update_g, balance_mode = args
    stores = [discriminator.store, recognizer.store, generator.store]
    saved = [(o.iterations if o is not None else 0) for o in opts]
    versions = None

    def roll_back():
        for o, it in zip(opts, saved):
            if o is not None:
                o.iterations = it
        if versions is not None:
            # the captured Adam launches keep the mirrors current: versions only matter for changes made OUTSIDE the graph
            for st, (v, wbv) in zip(stores, versions):
                st.version = v
                st.wb_version = wbv

    try:
        for st in stores:
            # every packed filter must be stale at capture time, so that the packing launches become part of the graph: a
            # forward pass since the last weight change (e.g. inference between two steps) would have left fresh entries,
            # the capture would skip the packs and every replay would then read filters from before its own Adam steps
            st.version += 1
            if rt.mode == "bf16":
                st.mirror(rt)                                   # fresh mirrors: no cast gets captured
        # optimizer state must exist BEFORE the capture: created inside it, the (m, v) slots would live in the graph's
        # private pool and their zero-fill would become a graph node (re-zeroing them on every replay)
        for o, st in ((opts[1], stores[0]), (opts[2], stores[1]), (opts[0], stores[2])):
            o.ensure_state(st)
        static = (rt.empty((b, 32, 16 * l_r, 1)), torch.zeros((b, l_r), device=rt.device, dtype=torch.int32),
                  torch.zeros((b, l_f), device=rt.device, dtype=torch.int32), rt.empty((b, latent_dim)))
        for t in static:
            t.zero_()
        versions = [(st.version, st.wb_version) for st in stores]
        torch.cuda.synchronize(rt.device)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=rt.device)
        n0 = rt.launch_count()
        if _graph_pool[0] is None:
            _graph_pool[0] = torch.cuda.graph_pool_handle()
        with torch.cuda.graph(graph, pool=_graph_pool[0], stream=side):
            rt.use_current_stream()
            stats = _step_device(rt, args, static[0], static[1], static[2], static[3], None)
        rt.use_current_stream()
        gs.launches = rt.launch_count() - n0
        rt.replayed_launches -= gs.launches                     # captured, not executed
        roll_back()
        gs.graph, gs.static, gs.stats = graph, static, stats
        gs.versions = [st.version for st in stores]
        gs.owners = (discriminator, recognizer, generator, opts)
    except Exception as ex:      # noqa: BLE001 -- capture is an optimisation: on any failure stay on the eager path
        import sys
        rt.use_current_stream()
        roll_back()
        gs.failed = True
        gs.graph = None
        print("scrabble-gan_b200: CUDA-graph capture of train_step failed ({}); staying eager".format(repr(ex)[:300]), file=sys.stderr)


def _replay(rt, gs, args, images, labels, fake_labels, noise):
    discriminator, recognizer, style_promoter, generator, opts, kind, balance, update_g, balance_mode = args
    stores = [discriminator.store, recognizer.store, generator.store]
    for i, st in enumerate(stores):
        if st.version != gs.versions[i]:                        # weights changed outside the graph (load / assign)
            if rt.mode == "bf16":
                st.mirror(rt)
            gs.versions[i] = st.version
    x_s, yr_s, yf_s, z_s = gs.static
    x_s.copy_(_as_tensor(images, np.float32).reshape(x_s.shape), non_blocking=True)
    yr_s.copy_(_as_tensor(labels, np.int32), non_blocking=True)
    yf_s.copy_(_as_tensor(fake_labels, np.int32), non_blocking=True)
    if noise is not None:
        z_s.copy_(_as_tensor(noise, np.float32), non_blocking=True)
    else:
        ops.random_(rt, z_s)
    used = [(opts[1], stores[0]), (opts[2], stores[1])] + ([(opts[0], stores[2])] if update_g else [])
    for o, _ in used:
        o.advance_for_replay(rt)
    gs.graph.replay()
    rt.replayed_launches += gs.launches
    # Python-side state the captured body would have advanced (the reference flips these flags at data_utils.py:449-466):
    # the Keras `trainable` flags as _step_device leaves them, and one store version per captured optimizer launch -- the
    # packed-filter caches of the layers key on it, so eager code after a replay re-packs from the CURRENT weights.  The
    # captured Adam launch wrote the bf16 mirror in the same pass, so the mirror stays in sync with the new version.
    discriminator.trainable = recognizer.trainable = not update_g
    for i, st in enumerate(stores):
        if any(s_ is st for _, s_ in used):
            mirror_current = st.wb is not None and st.wb_version == st.version
            st.version += 1
            if mirror_current:
                st.wb_version = st.version
            gs.versions[i] = st.version
    return gs.stats


def _step_device(rt, args, x_real, y_real, y_fake, g_in, style_imgs):
    """The device part of the step: every argument is a device tensor; returns the 16 statistics as a device tensor."""
    discriminator, recognizer, style_promoter, generator, opts, kind, apply_gradient_balance, update_g, balance_mode = args
    generator_optimizer, discriminator_optimizer, recognizer_optimizer, stylepromoter_optimizer = opts
    paper = bool(apply_gradient_balance) and balance_mode == "paper"
    use_w = style_promoter is not None
    b = y_real.shape[0]
    l_r, l_f = y_real.shape[1], y_fake.shape[1]
    # R's BatchNorm mode follows the Keras `trainable` flag at forward time (SURVEY Q5)
    recognizer.bn_training = bool(recognizer.trainable)
    # When the real and the fake words have the same length, D and R see both batches in ONE pass over a
    # [fake ; real] batch of 2B images (they have no cross-sample coupling: no batch-stat BN), which doubles the
    # GEMM M of every layer; G writes its tanh output straight into the first half, the real images are copied into
    # the second half.
    fused = (l_r == l_f) and not recognizer.bn_training
    if fused:
        xcat = rt.empty((2 * b, 32, 16 * l_r, 1))
        xcat[b:].copy_(x_real, non_blocking=True)
        x_real = xcat[b:]
        ycat = torch.empty((2 * b, l_r), device=rt.device, dtype=torch.int32)
        ycat[:b].copy_(y_fake)
        ycat[b:].copy_(y_real)
    assert g_in.shape[0] == b == y_fake.shape[0], "real and fake batches must have the same size (net_loss.py:49)"

    nets = [discriminator, recognizer, generator] + ([style_promoter] if use_w else [])
    for m in nets:
        m.store.zero_grad()
        m.sn_forward(rt, update_u=True)             # apply_sn: refresh W / sigma(W) (one power-iteration step, persistent u)
        if rt.use_tc:
            m.prepack(rt)                           # all forward filters of the network that the last Adam step made stale: one launch

    # ---- forward passes (data_utils.py:398-415) -------------------------------------------------------------------
    # D and R read the same images and share nothing else: R's passes go to the side stream (rt.branch) and run next to D's --
    # R's layers are small (most of its launches fill a fraction of the SMs), so they largely disappear inside D's time
    if fused:
        gen_images, g_cache = generator.forward(rt, g_in, y_fake, training=True, img_out=xcat[:b])
        br = rt.branch()
        with br:
            r_cat, rcc = recognizer.forward(rt, xcat, ycat)
        d_cat, dcc = discriminator.forward(rt, xcat)
        br.join()
        d_fake, d_real = d_cat.view(-1)[:b], d_cat.view(-1)[b:]
        r_fake, r_real = r_cat[:b], r_cat[b:]
    else:
        gen_images, g_cache = generator.forward(rt, g_in, y_fake, training=True)
        br = rt.branch()
        with br:
            r_fake, rfc = recognizer.forward(rt, gen_images, y_fake)
            r_real, rrc = recognizer.forward(rt, x_real, y_real)
        d_fake, dfc = discriminator.forward(rt, gen_images)
        d_real, drc = discriminator.forward(rt, x_real)
        br.join()
    s_fake = s_real = s_slot5 = None
    if use_w:
        s_fake, sfc = style_promoter.forward(rt, gen_images)
        s_real, src_c = style_promoter.forward(rt, style_imgs)
        if kind == net_loss.not_saturating.sg_kind:
            s_slot5, _ = style_promoter.forward(rt, x_real)      # dead code under hinge (SURVEY Q1): skipped there

    # ---- losses, gradient balancing, statistics (data_utils.py:418-442) -------------------------------------------
    sums = torch.empty(SG_LOSS_NSUMS, device=rt.device, dtype=torch.float64)
    call.sg_loss_sums(rt.ctx, kind, int(use_w), _p(d_real), _p(d_fake), _p(s_real), _p(s_fake), _p(s_slot5), _p(r_fake),
                      _p(r_real), b, _p(sums))
    rt.allreduce_small_(sums)
    ups = rt.empty((8, b))
    stats = rt.empty((16,))
    # rows 0,1 = (up_d_fake_d, up_d_real): adjacent and in [fake ; real] order for the fused D backward
    up_d_fake_d, up_d_real, up_s_real, up_s_fake_w, _up_s5, up_d_fake_g, up_s_fake_g, up_r_fake_g = ups
    call.sg_loss_finish(rt.ctx, kind, int(use_w), int(bool(apply_gradient_balance) and not paper), 1.0, _p(d_real), _p(d_fake), _p(s_real),
                        _p(s_fake), _p(s_slot5), _p(r_fake), b, _p(sums), _p(up_d_real), _p(up_d_fake_d), _p(up_s_real),
                        _p(up_s_fake_w), _p(_up_s5), _p(up_d_fake_g), _p(up_s_fake_g), _p(up_r_fake_g), _p(stats))

    # ---- D, R, W gradients (data_utils.py:449-459) ----------------------------------------------------------------
    # Data parallel: each network's flat gradient bucket is SUM-all-reduced (not averaged: SURVEY Q7) as soon as its
    # filter gradients are complete, on NCCL's stream, overlapping with the backward passes that follow.
    pending = []
    discriminator.trainable = True
    recognizer.trainable = True
    br = rt.branch()                     # R's backward (side stream) next to D's two backward passes (main stream)
    if fused:
        with br:
            if update_g:
                # ONE backward pass of R over the fused batch: filter gradients from the real half (R-loss, weight 1), image
                # gradient of the fake half with the G-loss per-sample weights (different samples: nothing mixes)
                dimg_r = recognizer.backward(rt, rcc, up_r_fake_g, wgrad=True, want_dx=True, wgrad_rows=(b, 2 * b), up_rows=(0, b))[:b]
            else:
                recognizer.backward(rt, recognizer.slice_cache(rcc, b, 2 * b), None, wgrad=True, want_dx=False)
            pending.append((id(recognizer), rt.allreduce_async_(recognizer.store.g, store=recognizer.store)))
        d_cache, d_up = dcc, ups[0:2].view(-1)
    else:
        with br:
            recognizer.backward(rt, rrc, None, wgrad=True, want_dx=False)
            pending.append((id(recognizer), rt.allreduce_async_(recognizer.store.g, store=recognizer.store)))
            if update_g:
                # R's image gradient of the fake batch (frozen R, G loss) right away: D's filter gradients queue up behind it
                # on the side stream, and G's backward pass must not wait for those
                dimg_r = recognizer.backward(rt, rfc, up_r_fake_g, wgrad=False, want_dx=True)
        discriminator.backward(rt, drc, up_d_real, wgrad=True, want_dx=False)
        d_cache, d_up = dfc, up_d_fake_d             # unfused: the merged pass below sees only the fake batch
    if update_g:
        # ONE backward pass of D for both losses (Discriminator.backward_merged); its filter gradients run on the side stream
        # next to the input-gradient chain and -- on one replica without spectral norm, where nothing reads D's bucket before
        # D's optimizer launch (side stream too) -- next to G's backward pass as well
        d_side = []
        dimg = discriminator.backward_merged(rt, d_cache, d_up, b, up_d_fake_g, 1.0, side=d_side)
        if rt.world_size > 1 or discriminator.store.sn is not None:
            rt.branch().join()
            d_side = None
    else:
        discriminator.backward(rt, d_cache, d_up, wgrad=True, want_dx=False)
    discriminator.sn_backward(rt)
    pending.append((id(discriminator), rt.allreduce_async_(discriminator.store.g, store=discriminator.store)))
    if use_w:
        style_promoter.trainable = True
        style_promoter.backward(rt, src_c, up_s_real, wgrad=True, want_dx=False)
        style_promoter.backward(rt, sfc, up_s_fake_w, wgrad=True, want_dx=False)
        style_promoter.sn_backward(rt)
        pending.append((id(style_promoter), rt.allreduce_async_(style_promoter.store.g, store=style_promoter.store)))

    # ---- optimizer steps (same call shape as the reference), each as soon as ITS bucket has been reduced -------------
    others = [(discriminator_optimizer, discriminator), (recognizer_optimizer, recognizer)]
    if use_w:
        others.append((stylepromoter_optimizer, style_promoter))

    # ---- G gradient through the frozen D, R (, W) (data_utils.py:462-468) -----------------------------------------
    if update_g:
        recognizer.trainable = False
        discriminator.trainable = False
        br.join()
        if use_w:
            style_promoter.trainable = False
            if kind == net_loss.hinge.sg_kind:
                dimg_w = style_promoter.backward(rt, sfc, up_s_fake_g, wgrad=False, want_dx=True)
                ops.axpby(rt, 1.0, dimg, 1.0, dimg_w, out=dimg)
        if paper:
            # gradient-level balancing (paper): grad_R <- alpha * std(grad_D) / std(grad_R) * grad_R on the image gradients,
            # population std over the GLOBAL batch (the five sums are all-reduced across replicas); the step's statistics
            # are patched with the balanced losses, alpha and the two stds
            bal = torch.empty(8, device=rt.device, dtype=torch.float64)
            call.sg_image_grad_balance_sums(rt.ctx, _p(dimg), _p(dimg_r), dimg.numel(), _p(bal))
            rt.allreduce_small_(bal)
            call.sg_image_grad_balance_apply(rt.ctx, _p(dimg), _p(dimg_r), dimg.numel(), 1.0, _p(bal), _p(dimg), _p(stats))
        else:
            ops.axpby(rt, 1.0, dimg, 1.0, dimg_r, out=dimg)
        # D, R (, W) are done with their weights: their optimizer launches (memory-bound) go to the side stream and run
        # under G's backward pass (compute- and latency-bound) instead of after it
        bo = rt.branch()
        with bo:
            _apply_all(rt, pending, others)
        generator.backward(rt, g_cache, dimg)
        generator.sn_backward(rt)
        if not rt.diag_skip_g_bucket:
            pending.append((id(generator), rt.allreduce_async_(generator.store.g, store=generator.store, exposed=True)))
        bo.join()
        _apply_all(rt, pending, [(generator_optimizer, generator)])
    else:
        br.join()
        _apply_all(rt, pending, others)
    return stats


def _apply_all(rt, pending, order):
    """optimizer.apply_gradients(zip(grads, trainable_variables)) per network (data_utils.py:452-468), each after the
    all-reduce of ITS gradient bucket (data parallel) has been ordered before the current stream."""
    work = dict(pending)
    for opt, model in order:
        w = work.get(id(model))
        if w is not None:
            w.wait()
        tv = model.store.trainable_variables
        opt.apply_gradients(zip([v.grad for v in tv], tv))


def generate_and_save_images(model, epoch, test_input, gen_path, char_vector):
    """Reference data_utils.py:493-519: G forward with training=False, (x+1)/2, dumped to disk (an .npy of the batch;
    a PNG grid as well when matplotlib is importable)."""
    predictions = model(test_input, training=False)
    predictions = ((predictions + 1) / 2.0).cpu().numpy()
    labels = np.asarray(test_input[1])
    os.makedirs(gen_path, exist_ok=True)
    np.save(os.path.join(gen_path, 'image_at_epoch_{:04d}.npy'.format(epoch)), predictions)
    try:
        import matplotlib
        matplotlib.use("Agg")
        import matplotlib.pyplot as plt
        for i in range(min(predictions.shape[0], 16)):
            plt.subplot(4, 4, i + 1)
            plt.imshow(predictions[i, :, :, 0], cmap='gray')
            plt.text(0, -1, "".join([char_vector[int(l)] for l in labels[i]]))
            plt.axis('off')
        plt.savefig(os.path.join(gen_path, 'image_at_epoch_{:04d}.png'.format(epoch)))
        plt.close()
    except Exception:
        pass
    return predictions


def train(dataset, generator, discriminator, recognizer, style_promoter, composite_gan, checkpoint, checkpoint_prefix,
          generator_optimizer, discriminator_optimizer, recognizer_optimizer, stylepromoter_optimizer, my_imgs, seed_labels,
          buffer_size, batch_size, epochs, model_path, latent_dim, gen_path, loss_fn, disc_iters, apply_gradient_balance,
          random_words, bucket_size, char_vector):
    """Thin re-use of the reference's training shell (data_utils.py:198-352): same 26 positional arguments, same
    summary-file columns, per-epoch save_weights of G and R.  `dataset` is any iterator of (images, labels)."""
    generator_save_dir = os.path.join(checkpoint_prefix, 'generator/')
    recognizer_save_dir = os.path.join(checkpoint_prefix, 'recognizer/')
    os.makedirs(generator_save_dir, exist_ok=True)
    os.makedirs(recognizer_save_dir, exist_ok=True)
    os.makedirs(gen_path, exist_ok=True)
    batch_per_epoch = int(buffer_size / batch_size) + 1
    rt_ = generator.rt
    if os.environ.get("SGAN_NO_PREFETCH", "0") != "1" and not isinstance(dataset, DevicePrefetcher):
        dataset = DevicePrefetcher(dataset, rt_)           # H2D of batch i+1 overlaps step i
    header = "disc_loss;disc_loss_real;disc_loss_fake;r_loss_real;r_loss_fake;r_loss_balanced;g_loss;g_lossT;g_lossS;" \
             "g_loss_final;alpha;r_loss_fake_std;g_loss_std;s_loss;s_loss_real;s_loss_fake\n"
    order = ("d_loss", "d_loss_real", "d_loss_fake", "r_loss_real", "r_loss_fake", "r_loss_balanced", "g_loss", "g_loss_added",
             "g_loss_balanced", "g_loss_final", "alpha", "r_loss_fake_std", "g_loss_std", "s_loss", "s_loss_real", "s_loss_fake")
    with open(os.path.join(gen_path, "batch_summary.txt"), "w") as batch_summary, \
            open(os.path.join(gen_path, "epoch_summary.txt"), "w") as epoch_summary:
        epoch_summary.write(header)
        batch_summary.write(header)
        for epoch_idx in range(epochs):
            start = time.time()
            totals = dict.fromkeys(STAT_NAMES, 0.0)
            for batch_idx in range(batch_per_epoch):
                image_batch, label_batch = next(dataset)
                my_img_batch = random.choices(my_imgs, k=batch_size) if my_imgs is not None else None
                out = train_step(epoch_idx, batch_idx, batch_per_epoch, image_batch, label_batch, discriminator, recognizer,
                                 style_promoter, composite_gan, generator_optimizer, discriminator_optimizer,
                                 recognizer_optimizer, stylepromoter_optimizer, my_img_batch, batch_size, latent_dim, loss_fn,
                                 disc_iters, apply_gradient_balance, random_words, bucket_size, gen_path)
                st = dict(zip(STAT_NAMES, out))
                batch_summary.write(";".join(str(st[k]) for k in order) + "\n")
                for k in STAT_NAMES:
                    totals[k] += st[k]
            epoch_summary.write(";".join(str(totals[k] / batch_per_epoch) for k in order) + "\n")
            if seed_labels is not None:
                generate_and_save_images(generator, epoch_idx + 1, seed_labels, gen_path, char_vector)
            print('Time for epoch {} is {} sec'.format(epoch_idx + 1, time.time() - start))
            generator.save_weights(os.path.join(generator_save_dir, str(epoch_idx + 1), 'cktp-' + str(epoch_idx + 1)))
            recognizer.save_weights(os.path.join(recognizer_save_dir, str(epoch_idx + 1), 'cktp-' + str(epoch_idx + 1)))

# ----------------------------------------------------------------------------------------------------
# input pipeline: length-bucketed batches staged through pinned memory, H2D copy overlapped with the running step
# ----------------------------------------------------------------------------------------------------
class DevicePrefetcher:
    """Wraps a generator with the interface of the reference's `load_prepare_data` (data_utils.py:14-84: an endless Python
    generator of (image_batch (B,32,16*len,1) float32, label_batch (B,len) int32), ONE length bucket per batch).  A worker
    thread pulls batch i+1, stages it in page-locked host memory (a small rotating pool per bucket shape) and copies it to
    the GPU on its own CUDA stream while step i runs; `next()` makes the compute stream wait on the copy's event and hands
    out DEVICE tensors, so train_step's own H2D copy disappears from the step.  (torch streams / events are plumbing.)"""

    def __init__(self, dataset, rt: Runtime, depth: int = 2):
        import queue
        import threading
        self.rt, self.depth = rt, max(int(depth), 1)
        self._src = iter(dataset)
        self._q = queue.Queue(maxsize=self.depth)
        self._stream = torch.cuda.Stream(device=rt.device)
        self._pool = {}
        self._live = None
        self._stop = False
        self._thread = threading.Thread(target=self._work, daemon=True)
        self._thread.start()

    def _pinned(self, shape, dtype, slot):
        key = (tuple(shape), dtype, slot)
        t = self._pool.get(key)
        if t is None:
            t = self._pool[key] = torch.empty(shape, dtype=dtype).pin_memory()
        return t

    def _work(self):
        torch.cuda.set_device(self.rt.device)
        slot = 0
        try:
            for images, labels in self._src:
                if self._stop:
                    return
                img = _as_tensor(images, np.float32)
                lab = _as_tensor(labels, np.int32)
                if img.is_cuda:
                    self._q.put((img, lab.to(self.rt.device), None))
                    continue
                # a pinned staging buffer may only be reused once its previous copy has been consumed: depth + 2 slots
                ph = self._pinned(img.shape, torch.float32, slot)
                pl = self._pinned(lab.shape, torch.int32, slot)
                slot = (slot + 1) % (self.depth + 2)
                ph.copy_(img)
                pl.copy_(lab)
                with torch.cuda.stream(self._stream):
                    d_img = ph.to(self.rt.device, non_blocking=True)
                    d_lab = pl.to(self.rt.device, non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(self._stream)
                self._q.put((d_img, d_lab, ev))
        except Exception as ex:      # noqa: BLE001 -- surfaced to the consumer
            self._q.put(ex)
        self._q.put(StopIteration())

    def __iter__(self):
        return self

    def __next__(self):
        item = self._q.get()
        if isinstance(item, StopIteration):
            raise StopIteration
        if isinstance(item, Exception):
            raise item
        d_img, d_lab, ev = item
        if ev is not None:
            torch.cuda.current_stream(self.rt.device).wait_event(ev)
            # the tensors were allocated on the copy stream: tell the caching allocator the compute stream uses them too
            d_img.record_stream(torch.cuda.current_stream(self.rt.device))
            d_lab.record_stream(torch.cuda.current_stream(self.rt.device))
        self._live = (d_img, d_lab)
        return d_img, d_lab

    def close(self):
        self._stop = True


def synthetic_word_batches_device(rt: Runtime, input_dim, batch_size, char_vector, bucket_size, bucket_weights=None, seed: int = 0):
    """Device-side synthetic loader with the interface of `load_prepare_data`: the bucket (word length) is drawn on the host
    from `bucket_weights` -- one bucket per batch, the reference's rule (data_utils.py:64) -- and the images / labels are
    generated directly in HBM by libsgan's Philox kernel (no host buffer, no H2D copy)."""
    h, _, c = input_dim
    rng = np.random.RandomState(seed)
    p = None
    if bucket_weights is not None:
        p = np.asarray(bucket_weights, np.float64)
        p = p / p.sum()
    n_chars = len(char_vector)
    while True:
        length = int(rng.choice(bucket_size, 1, p=p)[0]) + 1
        images = ops.random_(rt, rt.empty((batch_size, h, (h // 2) * length, c)), normal=False)
        u = ops.random_(rt, rt.empty((batch_size, length)), normal=False)
        labels = ((u + 1.0) * (0.5 * n_chars)).to(torch.int32).clamp_(0, n_chars - 1)      # (label synthesis only: not on the step)
        yield images, labels


# ----------------------------------------------------------------------------------------------------
# synthetic stand-ins for the reference's data loaders (the IAM dataset is not available here)
# ----------------------------------------------------------------------------------------------------
def synthetic_word_batches(input_dim, batch_size, char_vector, bucket_size, bucket_weights=None, seed: int = 0, pinned: bool = False):
    """Python generator with the interface of the reference's load_prepare_data (data_utils.py:14-84): yields
    (image_batch (B, h, (h/2)*len, c) float32 in [-1, 1], label_batch (B, len) int32), ONE random length bucket per batch
    drawn from `bucket_weights` (uniform if None) -- the reference's own rule (:64).  Images are uniform noise: this feeds
    benchmarks and the train() shell, it is not a dataset.  `pinned`: yield page-locked torch tensors (async H2D)."""
    h, _, c = input_dim
    rng = np.random.RandomState(seed)
    p = None
    if bucket_weights is not None:
        p = np.asarray(bucket_weights, np.float64)
        p = p / p.sum()
    while True:
        length = int(rng.choice(bucket_size, 1, p=p)[0]) + 1
        images = rng.uniform(-1.0, 1.0, size=(batch_size, h, (h // 2) * length, c)).astype(np.float32)
        labels = rng.randint(0, len(char_vector), size=(batch_size, length)).astype(np.int32)
        if pinned:
            yield torch.from_numpy(images).pin_memory(), torch.from_numpy(labels).pin_memory()
        else:
            yield images, labels


def synthetic_random_words(bucket_size, char_vector, words_per_bucket: int = 256, seed: int = 0):
    """Stand-in for load_random_word_list (data_utils.py:550-574): random_words[len-1] = list of encoded words of that length."""
    rng = np.random.RandomState(seed)
    return [[list(map(int, rng.randint(0, len(char_vector), size=length))) for _ in range(words_per_bucket)]
            for length in range(1, bucket_size + 1)]
