"""Model builders with the reference's signatures (src/bigacgan/net_architecture.py):
    make_recognizer(input_dim, sequence_length, output_classes, vis_model=True)                 reference :9-79
    make_generator(latent_dim, input_dim, embed_y, kernel_reg, blocks_with_attention, vocab_size, vis_model)  :182-296
    make_discriminator(input_dim, kernel_reg, blocks_with_attention, vis_model=True)            :299-355
    make_style_promoter(input_dim, kernel_reg, blocks_with_attention, vis_model=True)           :358-414
    make_gan(g_model, d_model, r_model, w_model, vis_model=True)                                 :531-561
    get_in_out_channels_gen / get_in_out_channels_disc                                          :565-586

The returned objects follow the protocol the reference's callers rely on (SURVEY.md section 8b): callable as
`model(inputs_list, training=bool)`, `.trainable` (settable), `.trainable_variables`, `.save_weights(prefix)`,
`.summary()`.  Internally each model has explicit forward/backward passes built from libsgan launches.

`kernel_reg` is accepted and stored but -- exactly as in the reference, where it is a Keras kernel_regularizer whose
loss nobody reads (SURVEY Q2) -- it does not change the forward pass or the gradients."""
from __future__ import annotations

import os
from typing import List, Optional

import numpy as np
import torch

from .. import ops
from .._abi import SG_F32, from_dlpack
from ..layers import BatchNormState, ConvLayer, DenseLayer, batch_stats
from ..params import ParamStore, init_glorot_uniform
from ..runtime import Runtime, get_runtime
from .arch_ops import NonLocalBlock, SpatialEmbedding
from .resnet_ops import ResNetBlockDown, ResNetBlockUp


# ----------------------------------------------------------------------------------------------------
# channel tables (reference :565-586)
# ----------------------------------------------------------------------------------------------------
def get_in_out_channels_gen(resolution=32):
    ch = 64
    if resolution == 32:
        channel_multipliers = [8, 4, 2, 1]
    else:
        raise ValueError("Unsupported resolution: {}".format(resolution))
    return [ch * c for c in channel_multipliers[:-1]], [ch * c for c in channel_multipliers[1:]]


def get_in_out_channels_disc(colors=1, resolution=32):
    ch = 64
    if colors not in [1, 3]:
        raise ValueError("Unsupported color channels: {}".format(colors))
    if resolution == 32:
        channel_multipliers = [1, 8, 16, 16]
    else:
        raise ValueError("Unsupported resolution: {}".format(resolution))
    out_channels = [ch * c for c in channel_multipliers]
    return [colors] + out_channels[:-1], out_channels


# ----------------------------------------------------------------------------------------------------
# input marshalling (host buffers / DLPack producers -> device tensors; plumbing only)
# ----------------------------------------------------------------------------------------------------
def _as_tensor(x, np_dtype):
    if isinstance(x, torch.Tensor):
        return x
    if isinstance(x, (list, tuple)) and len(x) > 0 and not np.isscalar(x[0]):
        x = np.stack([np.asarray(t.cpu() if isinstance(t, torch.Tensor) else t) for t in x], axis=0)
    if isinstance(x, (np.ndarray, list, tuple)):
        return torch.from_numpy(np.ascontiguousarray(np.asarray(x), dtype=np_dtype))
    return from_dlpack(x)


def to_device_f32(rt: Runtime, x) -> torch.Tensor:
    """Host numpy / pinned torch / device torch / DLPack producer -> contiguous fp32 tensor on the runtime's GPU."""
    return _as_tensor(x, np.float32).to(device=rt.device, dtype=torch.float32, non_blocking=True).contiguous()


def to_device_i32(rt: Runtime, x) -> torch.Tensor:
    return _as_tensor(x, np.int32).to(device=rt.device, dtype=torch.int32, non_blocking=True).contiguous()


def _nhwc(x: torch.Tensor) -> torch.Tensor:
    if x.dim() == 3:
        x = x.unsqueeze(-1)
    return x.contiguous()


class _Model:
    """Keras-like shell around a ParamStore."""

    def __init__(self, rt: Runtime, name: str, seed: int):
        self.rt = rt
        self.name = name
        self.store = ParamStore(rt, name, seed)
        self.trainable = True
        self.apply_sn = False

    def enable_spectral_norm(self, seed: int = 0):
        """Paper-faithful option `apply_sn` (SURVEY Q2 / Q3, section 8f): W / sigma(W) as a weight re-parameterisation with a
        persistent power-iteration vector u for every kernel the reference tags with kernel_regularizer=spectral_norm
        (resnet_ops.py:18-24,57-71,98-111; arch_ops.py:40-65; net_architecture.py:254,286,345): all conv / transposed conv /
        dense kernels of this model, i.e. every trainable variable named *.w except the filter bank.  In the reference the
        regulariser's value is never read, so the default (off) is the reference-faithful behaviour."""
        names = [v.name for v in self.store.vars if v.trainable and v.name.endswith(".w") and len(v.shape) >= 2]
        self.apply_sn = True
        return self.store.enable_spectral_norm(names, seed)

    def conv_layers(self):
        """Every ConvLayer / ConvTransposeLayer of the model (found by walking its attributes once)."""
        if getattr(self, "_conv_cache", None) is None:
            from ..layers import ConvLayer, ConvTransposeLayer
            found, seen = [], set()

            def walk(o, depth=0):
                if id(o) in seen or depth > 6:
                    return
                seen.add(id(o))
                if isinstance(o, (ConvLayer, ConvTransposeLayer)):
                    found.append(o)
                    return
                if isinstance(o, (list, tuple)):
                    for x in o:
                        walk(x, depth + 1)
                elif isinstance(o, dict):
                    for x in o.values():
                        walk(x, depth + 1)
                elif hasattr(o, "__dict__") and type(o).__module__.startswith("scrabble-gan_b200") and not isinstance(o, (ParamStore, Runtime)):
                    for x in vars(o).values():
                        walk(x, depth + 1)
            walk(self)
            self._conv_cache = found
        return self._conv_cache

    def prepack(self, rt) -> int:
        """After an optimizer step: re-pack all stale tensor-core filters of this model in one launch (layers.prepack)."""
        from ..layers import prepack
        return prepack(rt, self.conv_layers())

    def sn_forward(self, rt, update_u: bool) -> None:
        if self.apply_sn:
            self.store.sn.forward(rt, update_u)

    def sn_backward(self, rt) -> None:
        if self.apply_sn:
            self.store.sn.backward(rt)

    @property
    def trainable_variables(self):
        return self.store.trainable_variables if self.trainable else []

    @property
    def variables(self):
        return list(self.store.vars)

    def count_params(self) -> int:
        return self.store.n_trainable

    def summary(self):
        print('Model "{}": {:,} trainable parameters in {} variables'.format(self.name, self.store.n_trainable,
                                                                           len(self.store.trainable_variables)))

    def save_weights(self, prefix: str, save_format: Optional[str] = None) -> None:
        """Per-epoch checkpoint (reference data_utils.py:346-348: `model.save_weights(prefix)`).  Default: what Keras writes
        for such a prefix -- a TensorFlow checkpoint `<prefix>.index` + `<prefix>.data-00000-of-00001` whose keys are the
        reference model's `layer_with_weights-N/...` names (bigacgan/keras_names.py), so the file can be loaded by the
        reference; variables the reference does not track (the NonLocalBlock projections, SURVEY Q4) are stored under
        `_sgan/<name>`.  save_format="npz" (or a prefix ending in .npz): one .npz of every variable by libsgan name."""
        d = os.path.dirname(prefix)
        if d:
            os.makedirs(d, exist_ok=True)
        if save_format == "npz" or prefix.endswith(".npz"):
            path = prefix if prefix.endswith(".npz") else prefix + ".npz"
            np.savez(path, **{k: v.cpu().numpy() for k, v in self.store.state_dict().items()})
            return
        from .. import tf_checkpoint
        from . import keras_names
        keys = keras_names.keys_for(self)
        tensors = {}
        for name, t in self.store.state_dict().items():
            a = t.detach().cpu().numpy().astype(np.float32)
            if name in keys:
                tensors[keys[name]] = a.reshape(()) if name.endswith(".sigma") else a
            else:
                tensors["_sgan/" + name] = a
        tf_checkpoint.write_checkpoint(prefix, tensors)

    def load_weights(self, prefix: str, key_map=None) -> None:
        """Load a checkpoint written by `save_weights` -- or by the REFERENCE's `model.save_weights(prefix)` (TensorFlow
        checkpoint with Keras names; every tensor is shape-checked, `key_map` overrides derived names) -- or an .npz."""
        if os.path.exists(prefix + ".index"):
            from .. import tf_checkpoint
            from . import keras_names
            keras_names.load_keras_checkpoint(self, prefix, key_map=key_map)
            extra = {k[len("_sgan/"):]: v for k, v in tf_checkpoint.read_checkpoint(prefix).items() if k.startswith("_sgan/")}
            if extra:
                self.store.load_state_dict(extra, strict=False)
            return
        path = prefix if prefix.endswith(".npz") else prefix + ".npz"
        with np.load(path) as f:
            self.store.load_state_dict({k: f[k] for k in f.files})

    def state_dict(self):
        return self.store.state_dict()

    def load_state_dict(self, sd, strict=True):
        self.store.load_state_dict(sd, strict)


# ----------------------------------------------------------------------------------------------------
# ResNet-down trunk shared by D, the style promoter W and the in-G style encoder
# ----------------------------------------------------------------------------------------------------
class _DownTrunk:
    def __init__(self, store: ParamStore, prefix: str, colors: int, resolution: int, attention_after):
        in_ch, out_ch = get_in_out_channels_disc(colors=colors, resolution=resolution)
        self.blocks: List[ResNetBlockDown] = []
        self.attn = {}
        for i, (ci, co) in enumerate(zip(in_ch, out_ch)):
            name = "{}{}".format(prefix, i + 1)
            self.blocks.append(ResNetBlockDown(store, name, ci, co, i == len(in_ch) - 1))
            if attention_after(name):
                self.attn[i] = NonLocalBlock(store, name + ".attn", co)
        self.out_channels = out_ch[-1]

    def forward(self, rt: Runtime, x):
        caches = []
        net = x
        for i, blk in enumerate(self.blocks):
            net, c = blk.forward(rt, net)
            ca = None
            if i in self.attn:
                net, ca = self.attn[i].forward(rt, net)
            caches.append((c, ca))
        feats = ops.gap_relu_fwd(rt, net)                     # relu -> GlobalAveragePooling2D
        return feats, (caches, net)

    def backward(self, rt: Runtime, cache, dfeats, wgrad: bool, want_dx: bool, fake=None, side=None):
        """fake = (b, up, mult): merged backward (see ResNetBlockDown.backward); returns the image gradient of rows [0, b).
        side: list -- with `fake`, the blocks' filter gradients run on the side stream (their operands are collected here)."""
        caches, net = cache
        d = ops.gap_relu_bwd(rt, dfeats, net)
        for i in reversed(range(len(self.blocks))):
            c, ca = caches[i]
            if ca is not None:
                if fake is None:
                    d = self.attn[i].backward(rt, ca, d, wgrad)
                else:
                    # the non-local block interleaves its filter gradients with its input-gradient chain: rows [0, b) go
                    # through it twice -- with the constant weight (input gradient only), then, rescaled, with the whole
                    # batch for the filter gradients (whose input gradient is kept for the other rows only)
                    b, up, mult = fake
                    d_fake = self.attn[i].backward(rt, NonLocalBlock.slice_cache(ca, 0, b), d[:b].clone(), False)
                    ops.scale_samples_(rt, d[:b], up, mult)
                    d = self.attn[i].backward(rt, ca, d, wgrad)
                    d[:b].copy_(d_fake)
            d = self.blocks[i].backward(rt, c, d, wgrad, want_dx or i > 0, fake=fake, side=side)
        return d


class Discriminator(_Model):
    """make_discriminator / make_style_promoter: 4x ResNetBlockDown (64,512,1024,1024), NonLocalBlock after the
    blocks named in `blocks_with_attention`, ReLU, global average pool, Dense(1024 -> 1, no bias)."""

    def __init__(self, rt, input_dim, kernel_reg, blocks_with_attention, name="discriminator", seed=1, initialise=True):
        super().__init__(rt, name, seed)
        h, w, c = input_dim
        self.kernel_reg = kernel_reg
        self.trunk = _DownTrunk(self.store, "B", c, h, lambda nm: nm in blocks_with_attention)
        self.dense = DenseLayer(self.store, "dense", self.trunk.out_channels, 1)
        self.store.finalize(initialise)

    def forward(self, rt, x):
        feats, c = self.trunk.forward(rt, x)
        logits = self.dense.forward(rt, feats, x.shape[0])
        return logits, (feats, c)

    def backward(self, rt, cache, up, wgrad: bool = True, want_dx: bool = False):
        """up [n] = d(sum target)/d(logit).  Accumulates parameter gradients when wgrad; returns d/d(image) or None."""
        feats, c = cache
        n = feats.shape[0]
        dfeats = self.dense.backward(rt, feats, up, n, want_dx=True, wgrad=wgrad)
        return self.trunk.backward(rt, c, dfeats, wgrad, want_dx)

    def backward_merged(self, rt, cache, up_all, b: int, up_fake_g, mult: float, side):
        """ONE backward pass over a [fake ; real] batch that serves both the D loss and the G loss (data_utils.py:449-468
        differentiates them separately; frozen weights make the second tape the same linear map).  Back-propagation is linear
        in a sample's upstream weight, so rows [0, b) -- the fake images -- travel with the constant weight 1 / mult; the
        filter gradients of the D loss see them rescaled by up_all[i] * mult (hinge: exactly 0 or 1), and the image gradient
        of the G loss is the returned d/d(fake image) rescaled by up_fake_g[i] * mult.  up_all [2b] = d(D loss)/d(logit) for
        [fake ; real].  Accumulates D's parameter gradients; returns d(G loss)/d(fake images) [b, H, W, 1].
        side: a list -- the blocks' filter gradients are enqueued on the runtime's side stream and are complete only after the
        caller has joined it (rt.branch().join()); the list holds their operands and must stay alive until then."""
        feats, c = cache
        n = feats.shape[0]
        self.dense.backward(rt, feats, up_all, n, want_dx=False, wgrad=True)
        up_chain = up_all.clone()
        up_chain[:b].fill_(1.0 / mult)
        dfeats = self.dense.backward(rt, feats, up_chain, n, want_dx=True, wgrad=False)
        dimg = self.trunk.backward(rt, c, dfeats, True, True, fake=(b, up_all, mult), side=side)
        ops.scale_samples_(rt, dimg, up_fake_g, mult)
        return dimg

    def __call__(self, inputs, training=True):
        x = inputs[0] if isinstance(inputs, (list, tuple)) else inputs
        x = _nhwc(to_device_f32(self.rt, x))
        self.sn_forward(self.rt, update_u=False)
        logits, _ = self.forward(self.rt, x)
        return logits


# ----------------------------------------------------------------------------------------------------
# recogniser (CRNN + CTC)
# ----------------------------------------------------------------------------------------------------
class Recognizer(_Model):
    """conv64-pool22-conv128-pool22-conv256-conv256-pool21-conv512-BN-conv512-BN-pool21-conv512(2x2 valid) ->
    (B, 4L-1, 512) -> Dense softmax -> K.ctc_batch_cost; the model output IS the loss (B,1).  Keras default
    initialisers (glorot-uniform, zero bias).  BatchNorm runs in inference mode (`bn_training=False`) exactly as in
    the reference's train_step, where R.trainable is False during every forward pass (SURVEY Q5)."""

    def __init__(self, rt, input_dim, sequence_length, output_classes, name="recognizer", seed=3, initialise=True):
        super().__init__(rt, name, seed)
        h, w, c = input_dim
        assert h == 32, "the CRNN collapses exactly 32 rows to 1"
        self.output_classes = output_classes
        self.sequence_length = sequence_length
        chans = [(c, 64, 3, "same"), (64, 128, 3, "same"), (128, 256, 3, "same"), (256, 256, 3, "same"), (256, 512, 3, "same"),
                 (512, 512, 3, "same"), (512, 512, 2, "valid")]
        self.convs = [ConvLayer(self.store, "conv{}".format(i + 1), k, k, ci, co, pad, init=init_glorot_uniform)
                      for i, (ci, co, k, pad) in enumerate(chans)]
        self.bn5 = BatchNormState(self.store, "bn5", 512, affine=True)
        self.bn6 = BatchNormState(self.store, "bn6", 512, affine=True)
        self.dense = DenseLayer(self.store, "dense", 512, output_classes, use_bias=True, init=init_glorot_uniform)
        self.bn_training = False
        self.store.finalize(initialise)

    def _bn_forward(self, rt, x, bn: BatchNormState, out_dt, training: bool):
        if training:
            mean, rstd, count = batch_stats(rt, x, bn)
        else:
            mean, rstd = ops.bn_infer_prepare(rt, bn.moving_mean.data, bn.moving_var.data)
            count = 1
        y = ops.bn_apply(rt, x, mean, rstd, bn.gamma.data, bn.beta.data, False, False, out_dt)
        return y, (mean, rstd, count, training)

    def _bn_backward(self, rt, bn: BatchNormState, bc, dy, x, wgrad, out_dt, rows=None):
        """dy = grad of the BN output (fp32); x = BN input = relu(conv) (fp32).  Returns grad w.r.t. the conv
        pre-activation in the operand dtype (gated by x > 0).  `rows` = (a, b): samples whose parameter gradients count."""
        mean, rstd, count, training = bc
        s1, s2 = ops.bn_bwd_reduce(rt, dy, None, x, mean, rstd)
        if wgrad:
            a, b = rows if rows is not None else (0, s1.shape[0])
            ops.colsum_into(rt, s2[a:b], bn.c, bn.gamma.grad, accumulate=1)
            ops.colsum_into(rt, s1[a:b], bn.c, bn.beta.grad, accumulate=1)
        ab = None
        if training:
            ab = ops.bn_bwd_combine(rt, s1, s2, bn.gamma.data, False)
            rt.allreduce_small_(ab)
        return ops.bn_bwd_apply(rt, dy, None, x, mean, rstd, bn.gamma.data, False, ab, count, training, True, out_dt)

    def forward(self, rt, x, labels, want_grad: bool = True, input_length=None, label_length=None):
        """x (n,32,W,1) fp32, labels (n,L) int32 -> CTC loss (n,) plus a cache for backward.  input_length / label_length
        (n,) int32: a RAGGED batch exactly as the reference model takes one (its inputs are [images, labels, input_length,
        label_length], net_architecture.py:66-75): words of different lengths padded to a common width, every sample's CTC
        recursion over its own 4*len-1 frames and len labels."""
        logits, trunk = self._logits(rt, x, self.bn_training)
        loss, glogits = ops.ctc(rt, logits, labels, want_grad, input_length, label_length)
        return loss, trunk + (glogits,)

    def _logits(self, rt, x, bn_training: bool):
        """CRNN trunk + Dense pre-activations (n, W/4-1, classes) fp32, and the activations backward needs."""
        T = rt.op_dt
        cv = self.convs
        a1 = cv[0].forward(rt, x, relu=True, out_dt=T)
        p1 = ops.maxpool_fwd(rt, a1, 2, 2)
        a2 = cv[1].forward(rt, p1, relu=True, out_dt=T)
        p2 = ops.maxpool_fwd(rt, a2, 2, 2)
        a3 = cv[2].forward(rt, p2, relu=True, out_dt=T)
        a4 = cv[3].forward(rt, a3, relu=True, out_dt=T)
        p4 = ops.maxpool_fwd(rt, a4, 2, 1)
        a5 = cv[4].forward(rt, p4, relu=True, out_dt=SG_F32)
        b5, bc5 = self._bn_forward(rt, a5, self.bn5, T, bn_training)
        a6 = cv[5].forward(rt, b5, relu=True, out_dt=SG_F32)
        b6, bc6 = self._bn_forward(rt, a6, self.bn6, T, bn_training)
        p6 = ops.maxpool_fwd(rt, b6, 2, 1)
        a7 = cv[6].forward(rt, p6, relu=True, out_dt=SG_F32)           # (n, 1, W/4-1, 512)
        n, _, t, c = a7.shape
        logits = self.dense.forward(rt, a7, n * t).view(n, t, self.output_classes)
        return logits, (x, a1, p1, a2, p2, a3, a4, p4, a5, b5, bc5, a6, b6, bc6, p6, a7)

    def frame_probs(self, images) -> torch.Tensor:
        """Per-frame class probabilities (B, W/4-1, classes) fp32 on the device: the output of the reference model's Dense
        softmax layer (net_architecture.py:55), the input of K.ctc_decode.  BatchNorm always uses the moving statistics
        (inference); `bn_training` and the moving statistics are neither read nor changed.  images: (B, 32, W[, 1]) host
        buffer, device tensor or DLPack producer."""
        x = _nhwc(to_device_f32(self.rt, images))
        self.sn_forward(self.rt, update_u=False)
        logits, _ = self._logits(self.rt, x, bn_training=False)
        return ops.softmax_rows(self.rt, logits)

    @staticmethod
    def slice_cache(cache, a: int, b: int):
        x, a1, p1, a2, p2, a3, a4, p4, a5, b5, bc5, a6, b6, bc6, p6, a7, glogits = cache
        sl = lambda t: t[a:b]
        return (sl(x), sl(a1), sl(p1), sl(a2), sl(p2), sl(a3), sl(a4), sl(p4), sl(a5), sl(b5), bc5, sl(a6), sl(b6), bc6, sl(p6),
                sl(a7), sl(glogits) if glogits is not None else None)

    def backward(self, rt, cache, up, wgrad: bool = True, want_dx: bool = False, wgrad_rows=None, up_rows=None):
        """up [n] (or None = 1): per-sample upstream weight of the CTC loss.  `up_rows` = (a, b) applies `up` to those samples
        only (the others keep weight 1); `wgrad_rows` = (a, b) restricts the PARAMETER gradients to those samples -- together
        they let ONE pass over the fused [fake ; real] batch serve the R-loss update (real half, filter gradients) and
        the G-loss image gradient (fake half, per-sample weights): different samples, so the two never mix."""
        x, a1, p1, a2, p2, a3, a4, p4, a5, b5, bc5, a6, b6, bc6, p6, a7, glogits = cache
        T = rt.op_dt
        cv = self.convs
        n, _, t, c = a7.shape
        wa, wb = wgrad_rows if wgrad_rows is not None else (0, n)
        sl = lambda v: v[wa:wb]
        if up is not None:
            ua, ub = up_rows if up_rows is not None else (0, n)
            ops.scale_rows_(rt, glogits[ua:ub], up)                   # chain the per-sample upstream weight (None = 1)
        da7 = self.dense.backward(rt, a7, glogits, n * t, want_dx=True, wgrad=False).view(a7.shape)
        if wgrad:
            self.dense.backward(rt, sl(a7), sl(glogits), (wb - wa) * t, want_dx=False, wgrad=True)
        d7 = ops.mask_mul(rt, da7, a7, T)
        if wgrad:
            cv[6].wgrad(rt, sl(p6), sl(d7))
        dp6 = cv[6].dgrad(rt, d7, (p6.shape[1], p6.shape[2]))
        db6 = ops.maxpool_bwd(rt, dp6, b6, 2, 1, False, SG_F32)
        d6 = self._bn_backward(rt, self.bn6, bc6, db6, a6, wgrad, T, (wa, wb))
        if wgrad:
            cv[5].wgrad(rt, sl(b5), sl(d6))
        db5 = cv[5].dgrad(rt, d6, (b5.shape[1], b5.shape[2]))
        d5 = self._bn_backward(rt, self.bn5, bc5, db5, a5, wgrad, T, (wa, wb))
        if wgrad:
            cv[4].wgrad(rt, sl(p4), sl(d5))
        dp4 = cv[4].dgrad(rt, d5, (p4.shape[1], p4.shape[2]))
        d4 = ops.maxpool_bwd(rt, dp4, a4, 2, 1, True, T)
        if wgrad:
            cv[3].wgrad(rt, sl(a3), sl(d4))
        d3 = cv[3].dgrad(rt, d4, (a3.shape[1], a3.shape[2]), mask=a3, out_dt=T)
        if wgrad:
            cv[2].wgrad(rt, sl(p2), sl(d3))
        dp2 = cv[2].dgrad(rt, d3, (p2.shape[1], p2.shape[2]))
        d2 = ops.maxpool_bwd(rt, dp2, a2, 2, 2, True, T)
        if wgrad:
            cv[1].wgrad(rt, sl(p1), sl(d2))
        dp1 = cv[1].dgrad(rt, d2, (p1.shape[1], p1.shape[2]))
        d1 = ops.maxpool_bwd(rt, dp1, a1, 2, 2, True, T)
        if wgrad:
            cv[0].wgrad(rt, sl(x), sl(d1))
        if not want_dx:
            return None
        return cv[0].dgrad(rt, d1, (x.shape[1], x.shape[2]))

    def __call__(self, inputs, training=True):
        imgs, labels = inputs[0], inputs[1]
        x = _nhwc(to_device_f32(self.rt, imgs))
        y = to_device_i32(self.rt, labels)
        # [images, labels, input_length, label_length] as in the reference; with two inputs the lengths are implied
        # (T = W/4 - 1, L = labels.shape[1])
        il = to_device_i32(self.rt, inputs[2]).reshape(-1) if len(inputs) > 2 and inputs[2] is not None else None
        ll = to_device_i32(self.rt, inputs[3]).reshape(-1) if len(inputs) > 3 and inputs[3] is not None else None
        loss, _ = self.forward(self.rt, x, y, want_grad=False, input_length=il, label_length=ll)
        return loss.view(-1, 1)


# ----------------------------------------------------------------------------------------------------
# generator
# ----------------------------------------------------------------------------------------------------
class Generator(_Model):
    """Filter bank -> 3x ResNetBlockUp (512->256->128->64, CBN conditioned on z1..z3) -> NonLocalBlock after the
    blocks named in `blocks_with_attention` -> BN -> ReLU -> Conv3x3(64->1) -> tanh.
    Inputs: [z (B,128), y (B,L)] (upstream signature, the one run_inference.py:35 uses) or, with
    style_encoder=True, [style images (B,32,160,1), y] as in this fork (SURVEY Q8)."""

    def __init__(self, rt, latent_dim, input_dim, embed_y, kernel_reg, blocks_with_attention, vocab_size,
                 style_encoder: bool = False, name="generator", seed=2, initialise=True):
        super().__init__(rt, name, seed)
        h, w, c = input_dim
        in_ch, out_ch = get_in_out_channels_gen(h)
        self.num_blocks = len(in_ch)
        assert latent_dim % (self.num_blocks + 1) == 0 and latent_dim // (self.num_blocks + 1) == embed_y[0]
        self.latent_dim, self.zchunk = latent_dim, latent_dim // (self.num_blocks + 1)
        self.kernel_reg = kernel_reg
        self.colors = c
        self.embed = SpatialEmbedding(self.store, vocab_size, embed_y)
        self.blocks: List[ResNetBlockUp] = []
        self.attn = {}
        for i, (ci, co) in enumerate(zip(in_ch, out_ch)):
            nm = "B{}".format(i + 1)
            self.blocks.append(ResNetBlockUp(self.store, nm, ci, co, i == self.num_blocks - 1))
            if nm in blocks_with_attention:
                self.attn[i] = NonLocalBlock(self.store, nm + ".attn", co)
        self.bn = BatchNormState(self.store, "bn", out_ch[-1], affine=True)
        self.out = ConvLayer(self.store, "out", 3, 3, out_ch[-1], c)
        self.style = None
        if style_encoder:
            self.style = _DownTrunk(self.store, "B_style", c, h, lambda nm: nm == "B_style1")
            self.style_dense = DenseLayer(self.store, "style_dense", self.style.out_channels, latent_dim)
        self.store.finalize(initialise)

    def forward(self, rt, z_or_imgs, y, training: bool = True, img_out=None, ragged: bool = False):
        """ragged=True (inference only; SURVEY 8f rank 3): y is a label matrix padded with -1 on the right; every word is
        generated exactly as it would be alone at its own width 16 * len -- the inputs of all 3x3 convolutions are zeroed
        right of the word (its SAME padding), the non-local block leaves the keys beyond the word out of the softmax -- and
        the image is zero right of the word."""
        sc = None
        lens = None
        if ragged:
            if training:
                raise ValueError("ragged generator batches are an inference feature: batch-statistics BN couples the words of a batch")
            lens = ops.label_lengths(rt, y)
        if self.style is not None:
            feats, tc = self.style.forward(rt, z_or_imgs)
            z = self.style_dense.forward(rt, feats, feats.shape[0])
            sc = (feats, tc)
        else:
            z = z_or_imgs
        zs = self.latent_dim
        net, ec = self.embed.forward(rt, z, zs, y)
        # all 12 CBN gamma / beta Dense layers (resnet_ops.py:18-26) in ONE launch: [n, sum of 2 C] with per-layer column blocks
        segs = self._cbn_segments()
        gb_all = ops.cbn_dense_fwd(rt, z, zs, z.shape[0], [s[:3] for s in segs], self._cbn_wbase())
        gb, col = [], 0
        for c_, _, _, _ in segs:
            gb.append(gb_all[:, col:])
            col += c_
        gb_stride = gb_all.shape[1]
        caches = []
        for i, blk in enumerate(self.blocks):
            ragged = (lens, net.shape[2] // y.shape[1]) if lens is not None else None
            net, c = blk.forward(rt, net, training, (gb[4 * i], gb[4 * i + 1], gb_stride), (gb[4 * i + 2], gb[4 * i + 3], gb_stride),
                                 ragged)
            ca = None
            if i in self.attn:
                kv_cols = None
                if lens is not None:
                    kv_cols = lens * (net.shape[2] // y.shape[1] // 2)          # widths are even: no pooling window straddles a word's edge
                net, ca = self.attn[i].forward(rt, net, kv_cols=kv_cols)
            caches.append((c, ca))
        if training:
            mean, rstd, count = batch_stats(rt, net, self.bn)
        else:
            mean, rstd = ops.bn_infer_prepare(rt, self.bn.moving_mean.data, self.bn.moving_var.data)
            count = 1
        act = ops.bn_apply(rt, net, mean, rstd, self.bn.gamma.data, self.bn.beta.data, False, True, rt.op_dt)
        if lens is not None:
            ops.mask_width_(rt, act, lens, act.shape[2] // y.shape[1])
        pre = self.out.forward(rt, act)
        img = ops.tanh_fwd(rt, pre, img_out)
        if lens is not None:
            ops.mask_width_(rt, img.view(img.shape[0], img.shape[1], img.shape[2] // 4, 4) if img.shape[3] == 1 else img, lens,
                            (img.shape[2] // 4 if img.shape[3] == 1 else img.shape[2]) // y.shape[1])
        return img, (sc, z, ec, caches, net, mean, rstd, count, act, training, img)

    def backward(self, rt, cache, dimg):
        """Accumulates the gradients of all generator parameters for upstream d(target)/d(image) = dimg."""
        sc, z, ec, caches, net, mean, rstd, count, act, training, img = cache
        want_dz = self.style is not None
        n = net.shape[0]
        dpre = ops.tanh_bwd(rt, dimg, img)
        # filter gradients are off the input-gradient chain: on the side stream, next to the chain (ResNetBlockUp.backward)
        side = [dpre]
        with rt.branch():
            self.out.wgrad(rt, act, dpre)
        dact = self.out.dgrad(rt, dpre, (net.shape[1], net.shape[2]))
        s1, s2 = ops.bn_bwd_reduce(rt, dact, act, net, mean, rstd)
        ops.colsum_into(rt, s2, self.bn.c, self.bn.gamma.grad, accumulate=1)
        ops.colsum_into(rt, s1, self.bn.c, self.bn.beta.grad, accumulate=1)
        ab = None
        if training:
            ab = ops.bn_bwd_combine(rt, s1, s2, self.bn.gamma.data, False)
            rt.allreduce_small_(ab)
        d = ops.bn_bwd_apply(rt, dact, act, net, mean, rstd, self.bn.gamma.data, False, ab, count, training, False, SG_F32)
        dz = rt.zeros((n, self.latent_dim)) if want_dz else None
        defer = []
        for i in reversed(range(self.num_blocks)):
            c, ca = caches[i]
            if ca is not None:
                d = self.attn[i].backward(rt, ca, d, True)
            d = self.blocks[i].backward(rt, c, d, defer, side, dz[:, self.zchunk * (i + 1):] if want_dz else None, self.latent_dim)
        # the 12 Dense filter gradients dW = z_block^T @ (d gamma | d beta) in ONE launch
        by_layer = {id(cbn): (s1, s2) for cbn, s1, s2 in defer}
        segs, ups = [], []
        for (c_, zoff, woff, (cbn, which)) in self._cbn_segments(grad=True):
            s1, s2 = by_layer[id(cbn)]
            segs.append((c_, zoff, woff))
            ups.append(s2 if which == "gamma" else s1)
        ops.cbn_dense_wgrad(rt, z, self.latent_dim, n, segs, ups, self.store.g)
        self.embed.backward(rt, ec, d, dz, self.latent_dim)
        if want_dz:
            feats, tc = sc
            dfeats = self.style_dense.backward(rt, feats, dz, n, want_dx=True, wgrad=True)
            self.style.backward(rt, tc, dfeats, True, False)
        rt.branch().join()             # all filter gradients are in the bucket; only now may their operands be released
        side.clear()

    def _cbn_segments(self, grad: bool = False):
        """(C, column offset of the block's z slice, offset of the Dense kernel in the flat store, (layer, which)) for the
        12 gamma / beta Dense layers, in the order B1.cbn1.gamma, B1.cbn1.beta, B1.cbn2.gamma, ..."""
        out = []
        for i, blk in enumerate(self.blocks):
            for cbn in (blk.cbn1, blk.cbn2):
                for which, dense in (("gamma", cbn.gamma), ("beta", cbn.beta)):
                    out.append((cbn.c, self.zchunk * (i + 1), dense.w.offset, (cbn, which)))
        return out

    def _cbn_wbase(self):
        return self.store.w if self.store.w_eff is None else self.store.w_eff

    def __call__(self, inputs, training=True, ragged=None):
        """inputs = [z, y] (or [style images, y]).  A HOST label matrix that contains -1 padding is run as a ragged batch
        (see forward); for labels already on the device say ragged=True (no device read-back to find out)."""
        a, y = inputs[0], inputs[1]
        if ragged is None:
            host = isinstance(y, (np.ndarray, list, tuple)) or (isinstance(y, torch.Tensor) and not y.is_cuda)
            ragged = host and bool((np.asarray(y) < 0).any())
        y = to_device_i32(self.rt, y)
        if self.style is not None:
            a = _nhwc(to_device_f32(self.rt, a))
        else:
            a = to_device_f32(self.rt, a)
        self.sn_forward(self.rt, update_u=False)
        img, _ = self.forward(self.rt, a, y, training, ragged=bool(ragged))
        return img


class CompositeGAN(_Model):
    """make_gan: G followed by the frozen D, R (and W); returns [G(x), D(G(x)), R(G(x)), W(G(x))]."""

    def __init__(self, rt, g_model, d_model, r_model, w_model):
        self.rt = rt
        self.name = "composite_gan"
        self.generator, self.discriminator, self.recognizer, self.style_promoter = g_model, d_model, r_model, w_model
        self.store = g_model.store
        self.trainable = True

    @property
    def trainable_variables(self):
        # D, R, W are frozen inside the composite (reference :543-545): only G's variables are trainable here
        return self.generator.store.trainable_variables

    def __call__(self, inputs, training=True):
        a, y = inputs[0], inputs[1]
        img = self.generator([a, y], training=training)
        d = self.discriminator([img], training=training)
        r = self.recognizer([img, to_device_i32(self.rt, y)], training=training)
        w = self.style_promoter([img], training=training) if self.style_promoter is not None else None
        return [img, d, r, w]


# ----------------------------------------------------------------------------------------------------
# builders
# ----------------------------------------------------------------------------------------------------
def make_recognizer(input_dim, sequence_length, output_classes, vis_model=True, rt: Optional[Runtime] = None, seed: int = 3,
                    initialise: bool = True):
    """`initialise=False` (keyword extension, all builders): skip the random initialisation when the caller loads weights."""
    m = Recognizer(rt or get_runtime(), input_dim, sequence_length, output_classes, seed=seed, initialise=initialise)
    if vis_model:
        m.summary()
    return m


def make_generator(latent_dim, input_dim, embed_y, kernel_reg, blocks_with_attention, vocab_size, vis_model=True,
                   style_encoder: bool = False, rt: Optional[Runtime] = None, seed: int = 2, initialise: bool = True,
                   apply_sn: bool = False):
    m = Generator(rt or get_runtime(), latent_dim, input_dim, embed_y, kernel_reg, blocks_with_attention, vocab_size,
                  style_encoder=style_encoder, seed=seed, initialise=initialise)
    if apply_sn:
        m.enable_spectral_norm(seed)
    if vis_model:
        m.summary()
    return m


def make_discriminator(input_dim, kernel_reg, blocks_with_attention, vis_model=True, rt: Optional[Runtime] = None, seed: int = 1,
                       initialise: bool = True, apply_sn: bool = False):
    m = Discriminator(rt or get_runtime(), input_dim, kernel_reg, blocks_with_attention, "discriminator", seed, initialise)
    if apply_sn:
        m.enable_spectral_norm(seed)
    if vis_model:
        m.summary()
    return m


def make_style_promoter(input_dim, kernel_reg, blocks_with_attention, vis_model=True, rt: Optional[Runtime] = None, seed: int = 4,
                        initialise: bool = True, apply_sn: bool = False):
    m = Discriminator(rt or get_runtime(), input_dim, kernel_reg, blocks_with_attention, "style_promoter", seed, initialise)
    if apply_sn:
        m.enable_spectral_norm(seed)
    if vis_model:
        m.summary()
    return m


def make_gan(g_model, d_model, r_model, w_model=None, vis_model=True):
    d_model.trainable = False
    r_model.trainable = False
    if w_model is not None and not isinstance(w_model, str):
        w_model.trainable = False
    else:
        w_model = None          # the reference's main.py passes a path string here by mistake (SURVEY Q9)
    m = CompositeGAN(g_model.rt, g_model, d_model, r_model, w_model)
    if vis_model:
        m.summary()
    return m
