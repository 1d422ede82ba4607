"""BigGAN ResNet blocks with conditional batch-norm -- B200-native counterparts of the reference's
src/bigacgan/resnet_ops.py (ConditionalBatchNorm :5-33, ResNetBlockUp :36-81, ResNetBlockDown :84-120).

Every block exposes forward(rt, x, ...) -> (y, cache) and backward(rt, cache, dy, ...) -> dx with hand-derived
gradients; all arithmetic is libsgan launches.  Dtype discipline: the residual stream and every gradient that is
summed is fp32; tensors that are consumed only as convolution operands are written directly in the operand
dtype (bf16 in "bf16" mode) by the producing kernel's epilogue."""
from __future__ import annotations

from .. import ops
from .._abi import SG_F32
from ..layers import BatchNormState, ConvLayer, ConvTransposeLayer, DenseLayer, batch_stats
from ..params import ParamStore
from ..runtime import Runtime


class ConditionalBatchNorm:
    """BN(scale=False, center=False) batch statistics (eps 1e-3, momentum .99) then * gamma(z) + beta(z), with
    gamma, beta = Dense(32 -> C, no bias)(z); NOT 1 + gamma.  (reference resnet_ops.py:13-28)"""

    def __init__(self, store: ParamStore, name: str, c: int, zdim: int = 32):
        self.c = c
        self.gamma = DenseLayer(store, name + ".gamma", zdim, c)
        self.beta = DenseLayer(store, name + ".beta", zdim, c)
        self.bn = BatchNormState(store, name, c, affine=False)

    def forward(self, rt: Runtime, x, gb, training: bool, relu: bool, out_dt: int):
        """gb = (gamma, beta, row stride): views into the grouped Dense output of the whole generator (one launch for all
        CBN layers, ops.cbn_dense_fwd)."""
        if training:
            mean, rstd, count = batch_stats(rt, x, self.bn)
        else:
            mean, rstd = ops.bn_infer_prepare(rt, self.bn.moving_mean.data, self.bn.moving_var.data)
            count = 1
        g, b, gs = gb
        y = ops.bn_apply(rt, x, mean, rstd, g, b, True, relu, out_dt, gb_stride=gs)
        return y, (x, y if relu else None, mean, rstd, g, count, training, gs)

    def backward(self, rt: Runtime, cache, dy, defer, out_dt: int = SG_F32, out=None, accumulate: bool = False, dz_out=None,
                 dz_ld: int = 0):
        """dy: gradient w.r.t. the (post-ReLU) output.  Records (layer, d beta, d gamma) in the list `defer`, so that the caller
        computes the Dense weight gradients of all CBN layers in one grouped launch, and, when dz_out is given, adds d/dz into
        dz_out (row stride dz_ld).  Returns dx."""
        x, act, mean, rstd, g, count, training, gs = cache
        n = x.shape[0]
        s1, s2 = ops.bn_bwd_reduce(rt, dy, act, x, mean, rstd)          # s1 = d beta [n,c], s2 = d gamma [n,c]
        ab = None
        if training:
            ab = ops.bn_bwd_combine(rt, s1, s2, g, True, gb_stride=gs)
            rt.allreduce_small_(ab)                                           # sync-BN backward statistics
        dx = ops.bn_bwd_apply(rt, dy, act, x, mean, rstd, g, True, ab, count, training, False, out_dt, out, int(accumulate),
                              gb_stride=gs)
        defer.append((self, s1, s2))
        if dz_out is not None:
            ops.gemm(rt, s2, self.gamma.w.eff, n, self.gamma.cin, self.c, trans_b=True, out=dz_out, ldc=dz_ld, accumulate=1)
            ops.gemm(rt, s1, self.beta.w.eff, n, self.beta.cin, self.c, trans_b=True, out=dz_out, ldc=dz_ld, accumulate=1)
        return dx


class ResNetBlockUp:
    """CBN -> ReLU -> ConvT3x3(stride (2,2) | (2,1) for the last block) -> CBN -> ReLU -> Conv3x3, plus a
    ConvT1x1 shortcut of the same stride on the raw input (value only at even positions, bias everywhere).
    (reference resnet_ops.py:46-74)"""

    def __init__(self, store: ParamStore, name: str, ci: int, co: int, is_last_block: bool):
        self.name, self.ci, self.co = name, ci, co
        self.stride = (2, 1) if is_last_block else (2, 2)
        self.cbn1 = ConditionalBatchNorm(store, name + ".cbn1", ci)
        self.up = ConvTransposeLayer(store, name + ".up", 3, ci, co, self.stride)
        self.cbn2 = ConditionalBatchNorm(store, name + ".cbn2", co)
        self.conv = ConvLayer(store, name + ".conv", 3, 3, co, co)
        self.short = ConvTransposeLayer(store, name + ".short", 1, ci, co, self.stride)

    def forward(self, rt: Runtime, x, training: bool, gb1, gb2, ragged=None):
        """gb1, gb2: (gamma, beta, row stride) of cbn1 / cbn2 (ConditionalBatchNorm.forward).  ragged = (lens, columns per
        character of x): the inputs of both 3x3 convolutions are zeroed right of every word's own width, so a short word of a
        padded batch sees the zero padding it would see alone (inference only)."""
        a1, c1 = self.cbn1.forward(rt, x, gb1, training, True, rt.op_dt)
        if ragged is not None:
            ops.mask_width_(rt, a1, ragged[0], ragged[1])
        u = self.up.forward(rt, a1)
        a2, c2 = self.cbn2.forward(rt, u, gb2, training, True, rt.op_dt)
        if ragged is not None:
            ops.mask_width_(rt, a2, ragged[0], ragged[1] * self.stride[1])
        bsum = ops.axpby(rt, 1.0, self.conv.b.data, 1.0, self.short.b.data)      # conv bias + shortcut bias (everywhere)
        h = self.conv.forward(rt, a2, bias=bsum)
        xs = ops.cast(rt, x, rt.op_dt)
        self.short.forward(rt, xs, out=h, accumulate=True, bias=None)
        return h, (c1, c2, a1, a2, xs, x.shape)

    def backward(self, rt: Runtime, cache, dh, defer, side, dz_out=None, dz_ld: int = 0):
        """defer: list of the CBN layers' Dense gradient operands (ConditionalBatchNorm.backward).  side: a list -- the three
        filter gradients of the block are not on the input-gradient chain, so they are enqueued on the runtime's side stream
        (rt.branch) and run next to the chain's (small, latency-bound) kernels; the list collects the temporaries they read,
        which the caller keeps alive until it has joined the side stream."""
        c1, c2, a1, a2, xs, xshape = cache
        n, hh, ww, _ = xshape
        dh_op = ops.cast(rt, dh, rt.op_dt)

        def off_chain(fn, *keep):
            side.extend(keep)
            with rt.branch():
                fn()
        # main branch, back to front
        off_chain(lambda: self.conv.wgrad(rt, a2, dh_op, also_bias=self.short.b.grad), dh_op)   # the shortcut bias sees the same upstream gradient
        da2 = self.conv.dgrad(rt, dh_op, (hh * self.stride[0], ww * self.stride[1]))
        du = self.cbn2.backward(rt, c2, da2, defer, out_dt=rt.op_dt, dz_out=dz_out, dz_ld=dz_ld)
        off_chain(lambda: self.up.wgrad(rt, a1, du), du)
        da1 = self.up.dgrad(rt, du)
        dx = self.cbn1.backward(rt, c1, da1, defer, out_dt=SG_F32, dz_out=dz_out, dz_ld=dz_ld)
        # shortcut branch
        off_chain(lambda: self.short.wgrad(rt, xs, dh_op, bias_grad=False), dh_op)
        self.short.dgrad(rt, dh_op, out=dx, accumulate=True)
        return dx


class ResNetBlockDown:
    """ReLU -> Conv3x3 -> ReLU -> Conv3x3 -> [AvgPool2x2 unless last]; shortcut Conv1x1 on the RAW input ->
    [AvgPool]; add.  The leading ReLU is applied in every block, including the first one on raw images (Q11).
    avgpool(a) + avgpool(b) = avgpool(a + b), so the shortcut is accumulated into the main branch before ONE
    pooling pass.  (reference resnet_ops.py:93-115)"""

    def __init__(self, store: ParamStore, name: str, ci: int, co: int, is_last_block: bool):
        self.name, self.ci, self.co, self.is_last = name, ci, co, is_last_block
        self.conv1 = ConvLayer(store, name + ".conv1", 3, 3, ci, co)
        self.conv2 = ConvLayer(store, name + ".conv2", 3, 3, co, co)
        self.short = ConvLayer(store, name + ".short", 1, 1, ci, co)

    def forward(self, rt: Runtime, x):
        n, h, w, _ = x.shape
        narrow = self.ci < 32                       # image input: edge layer on the FFMA path, fp32 operands
        in_dt = SG_F32 if narrow else rt.op_dt
        xr, xs = ops.act_prep(rt, x, True, in_dt != SG_F32, in_dt)
        if xs is None:
            xs = x
        h1 = self.conv1.forward(rt, xr, relu=True, out_dt=rt.op_dt)
        h2 = None
        if not narrow and rt.use_tc:
            # conv2 and the 1x1 shortcut in ONE launch: the shortcut's k-blocks land in the same TMEM accumulator
            bsum = ops.axpby(rt, 1.0, self.conv2.b.data, 1.0, self.short.b.data)
            h2 = self.conv2.forward_with_shortcut(rt, h1, self.short, xs, bsum)
        if h2 is None and narrow and rt.use_tc and self.ci == 1:
            # one-channel input (the image): the 1x1 shortcut is an outer product, added in conv2's epilogue
            bsum = ops.axpby(rt, 1.0, self.conv2.b.data, 1.0, self.short.b.data)
            h2 = self.conv2.forward_with_rank1_shortcut(rt, h1, self.short, xs, bsum)
        if h2 is None:
            h2 = self.conv2.forward(rt, h1)
            self.short.forward(rt, xs, out=h2, accumulate=True)
        out = h2 if self.is_last else ops.avgpool2_fwd(rt, h2)
        return out, (xr, xs, h1, (h, w))

    def backward(self, rt: Runtime, cache, dout, wgrad: bool = True, want_dx: bool = True, fake=None, side=None):
        """fake = (b, up, mult) -- the merged discriminator backward (Discriminator.backward_merged): rows [0, b) of the batch
        carry a CONSTANT upstream weight through the input-gradient chain; the filter gradients need the per-sample weights
        up[i] * mult of the D loss instead, so the block first computes its input gradients from the unscaled tensors, then
        rescales rows [0, b) of the tensors the filter gradients read, in place.  With `fake`, dx is returned for rows [0, b)
        only (the image gradient of the real half is never needed)."""
        xr, xs, h1, (h, w) = cache
        dpre = ops.cast(rt, dout, rt.op_dt) if self.is_last else ops.avgpool2_bwd(rt, dout, rt.op_dt)
        if fake is None:
            if wgrad:
                # the shortcut bias sees the same upstream gradient as conv2's bias: one column sum serves both
                # (sum over pixels of avgpool_bwd(dout) == sum over pooled pixels of dout: read the 4x smaller fp32 tensor)
                self.conv2.wgrad(rt, h1, dpre, also_bias=self.short.b.grad, bias_src=dout)
                self.short.wgrad(rt, xs, dpre, bias_grad=False)
            dh1 = self.conv2.dgrad(rt, dpre, (h, w), mask=h1, out_dt=rt.op_dt)
            if wgrad:
                self.conv1.wgrad(rt, xr, dh1)
            if not want_dx:
                return None
            dx = self.conv1.dgrad(rt, dh1, (h, w), mask=xr)
            self.short.dgrad(rt, dpre, (h, w), out=dx, accumulate=True)
            return dx
        b, up, mult = fake
        dh1 = self.conv2.dgrad(rt, dpre, (h, w), mask=h1, out_dt=rt.op_dt)
        dx = None
        if want_dx:
            rows = slice(0, b) if self.ci < 32 else slice(None)          # first block: only the fake half's image gradient
            dx = self.conv1.dgrad(rt, dh1[rows], (h, w), mask=xr[rows])
            self.short.dgrad(rt, dpre[rows], (h, w), out=dx, accumulate=True)
        if wgrad:
            # off the input-gradient chain: the rescale and the three filter gradients go to the side stream (everything
            # the chain reads from these tensors has been enqueued above); the caller keeps the tensors alive until it joins
            side.extend((dpre, dh1, dout))
            with rt.branch():
                seen = set()
                for t in (dpre, dh1, dout):
                    if t.data_ptr() not in seen:             # last block in fp32 mode: dpre IS dout (no cast, no pooling)
                        seen.add(t.data_ptr())
                        ops.scale_samples_(rt, t[:b], up, mult)
                self.conv2.wgrad(rt, h1, dpre, also_bias=self.short.b.grad, bias_src=dout)
                self.short.wgrad(rt, xs, dpre, bias_grad=False)
                self.conv1.wgrad(rt, xr, dh1)
        return dx
