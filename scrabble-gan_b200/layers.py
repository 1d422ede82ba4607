"""Primitive layers with explicit forward / input-gradient / filter-gradient methods (no autograd, no tape).

A layer owns Variables in a ParamStore and caches (a) one sg_conv_desc per (role, shape, epilogue) and (b) the packed
tensor-core weight matrices, which are re-packed lazily when the store's version changes (i.e. after an optimizer
step or a weight load)."""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

from . import ops
from ._abi import SG_F32
from .params import ParamStore, Variable, init_ones, init_orthogonal, init_zeros
from .runtime import Runtime, dt_of


class ConvLayer:
    """tf.keras.layers.Conv2D(filters, (kh,kw), strides 1, padding same|valid, use_bias) -- HWIO kernel.
    Reference call sites: resnet_ops.py:65,98,103,109; net_architecture.py:28-49,283; arch_ops.py:38-65."""

    def __init__(self, store: ParamStore, name: str, kh: int, kw: int, ci: int, co: int, padding: str = "same",
                 use_bias: bool = True, init=init_orthogonal):
        self.kh, self.kw, self.ci, self.co, self.padding = kh, kw, ci, co, padding
        self.w: Variable = store.add(name + ".w", (kh, kw, ci, co), init)
        self.b: Optional[Variable] = store.add(name + ".b", (co,), init_zeros) if use_bias else None
        self.store = store
        self._descs: Dict[tuple, object] = {}
        self._packed: Dict[tuple, Tuple[int, torch.Tensor]] = {}

    # -- helpers --------------------------------------------------------------------------------------
    def out_hw(self, h: int, w: int) -> Tuple[int, int]:
        return (h, w) if self.padding == "same" else (h - self.kh + 1, w - self.kw + 1)

    def _desc(self, role: str, n, h, w, in_dt, out_dt, relu=0, accumulate=0, mask_dt=SG_F32):
        key = (role, n, h, w, in_dt, out_dt, relu, accumulate, mask_dt)
        d = self._descs.get(key)
        if d is None:
            if role == "fwd":
                d = ops.desc_conv_fwd(n, h, w, self.ci, self.co, self.kh, self.kw, self.padding, in_dt, out_dt, relu, accumulate,
                                      mask_dt)
            else:
                d = ops.desc_conv_dgrad(n, h, w, self.ci, self.co, self.kh, self.kw, self.padding, in_dt, out_dt, accumulate,
                                        mask_dt)
            self._descs[key] = d
        return d

    def _pack(self, rt: Runtime, role: str, d):
        if not ops.tc_ok(rt, d):
            return None
        key = (role, d.in_dt)
        ent = self._packed.get(key)
        if ent is None or ent[0] != self.store.version:
            buf = ent[1] if ent is not None else None
            buf = ops.pack_weights(rt, d, self.w.eff, buf)
            self._packed[key] = (self.store.version, buf, d)      # the descriptor lets layers.prepack() redo this in a batch
            return buf
        return ent[1]

    # -- compute --------------------------------------------------------------------------------------
    def forward(self, rt: Runtime, x: torch.Tensor, relu: bool = False, out_dt: int = SG_F32, out=None,
                accumulate: bool = False, bias="own") -> torch.Tensor:
        n, h, w, _ = x.shape
        d = self._desc("fwd", n, h, w, dt_of(x), out_dt if out is None else dt_of(out), int(relu), int(accumulate))
        if out is None:
            ho, wo = self.out_hw(h, w)
            out = rt.empty((n, ho, wo, self.co), out_dt)
        b = (self.b.data if self.b is not None else None) if isinstance(bias, str) else bias
        if ops.direct_ok(rt, d):
            ops.conv_run(rt, d, x, self.w.eff, None, b, None, out, w_mirror=self.w.mirror(rt))
        else:
            ops.conv_run(rt, d, x, self.w.eff, self._pack(rt, "fwd", d), b, None, out)
        return out

    def forward_with_shortcut(self, rt: Runtime, x: torch.Tensor, short: "ConvLayer", x2: torch.Tensor, bias, out_dt: int = SG_F32):
        """self(x) + short(x2) + bias in ONE tensor-core launch (short is a 1x1 conv; its k-blocks are accumulated into the
        same TMEM tile).  Returns None when the pair cannot take the tensor-core path (caller falls back)."""
        n, h, w, _ = x.shape
        d = self._desc("fwd", n, h, w, dt_of(x), out_dt, 0, 0)
        d2 = short._desc("fwd", n, h, w, dt_of(x2), out_dt, 0, 0)
        if short.kh != 1 or short.kw != 1 or dt_of(x) != dt_of(x2) or not (ops.tc_ok(rt, d) and ops.tc_ok(rt, d2)):
            return None
        ho, wo = self.out_hw(h, w)
        out = rt.empty((n, ho, wo, self.co), out_dt)
        ops.conv_run_dual(rt, d, x, self._pack(rt, "fwd", d), d2, x2, short._pack(rt, "fwd", d2), bias, None, out)
        return out

    def forward_with_rank1_shortcut(self, rt: Runtime, x: torch.Tensor, short: "ConvLayer", x2: torch.Tensor, bias, out_dt: int = SG_F32):
        """self(x) + short(x2) + bias in ONE tensor-core launch when short is a 1x1 conv of a ONE-channel fp32 tensor (the
        raw image): that conv is the outer product x2[p] * w[c], added in the epilogue.  None when not applicable."""
        n, h, w, _ = x.shape
        d = self._desc("fwd", n, h, w, dt_of(x), out_dt, 0, 0)
        if short.kh != 1 or short.kw != 1 or short.ci != 1 or short.co != self.co or dt_of(x2) != SG_F32 or not ops.tc_ok(rt, d) or \
                self.out_hw(h, w) != (h, w):
            return None
        out = rt.empty((n, h, w, self.co), out_dt)
        ops.conv_run_rank1(rt, d, x, self._pack(rt, "fwd", d), bias, None, out, x2, short.w.eff.view(-1))
        return out

    def dgrad(self, rt: Runtime, dy: torch.Tensor, in_hw: Tuple[int, int], mask=None, out_dt: int = SG_F32, out=None,
              accumulate: bool = False) -> torch.Tensor:
        n = dy.shape[0]
        h, w = in_hw
        odt = out_dt if out is None else dt_of(out)
        d = self._desc("dgrad", n, h, w, dt_of(dy), odt, 0, int(accumulate), dt_of(mask) if mask is not None else SG_F32)
        if out is None:
            out = rt.empty((n, h, w, self.ci), out_dt)
        if ops.direct_ok(rt, d):
            ops.conv_run(rt, d, dy, self.w.eff, None, None, mask, out, w_mirror=self.w.mirror(rt))
        else:
            ops.conv_run(rt, d, dy, self.w.eff, self._pack(rt, "dgrad", d), None, mask, out)
        return out

    def wgrad(self, rt: Runtime, x: torch.Tensor, dy: torch.Tensor, bias_grad: bool = True, also_bias=None, bias_src=None) -> None:
        """Filter (+ bias) gradient.  `also_bias`: a second bias gradient [co] that sees the same upstream gradient (the
        shortcut of a ResNet block): dy is column-summed ONCE and the sum is added to both.  `bias_src`: a tensor with the
        same column sums as dy that is cheaper to read (the un-pooled fp32 gradient: avg-pool backward preserves sums)."""
        n, h, w, _ = x.shape
        d = self._desc("fwd", n, h, w, dt_of(x), dt_of(dy))
        want_b = bias_grad and self.b is not None
        if ops.conv_wgrad(rt, d, x, dy, self.w.grad, db=self.b.grad if want_b else None, db2=also_bias if want_b else None):
            return                                        # bias gradient(s) came out of the same tensor-core launch
        if want_b:
            src = dy if bias_src is None else bias_src
            if also_bias is None:
                ops.colsum_into(rt, src, self.co, self.b.grad, accumulate=1)
            else:
                s = rt.empty((self.co,), SG_F32)
                ops.colsum_into(rt, src, self.co, s, accumulate=0)
                ops.axpby(rt, 1.0, s, 1.0, self.b.grad, out=self.b.grad)
                ops.axpby(rt, 1.0, s, 1.0, also_bias, out=also_bias)


def prepack(rt: Runtime, convs) -> int:
    """Re-pack, in ONE launch per 32 filters, every packed tensor-core filter of the given layers whose weights changed since
    it was packed (i.e. after an optimizer step): the per-layer lazy packing in ConvLayer._pack then finds fresh entries.
    Only filters that have been used before are known (their descriptor is cached with the packed buffer)."""
    import ctypes as C
    from . import _abi
    lib = _abi.load()
    jobs = []
    for lay in convs:
        ver = lay.store.version
        for key, ent in lay._packed.items():
            if ent[0] == ver or len(ent) < 3:
                continue
            d, buf = ent[2], ent[1]
            src = lay.w.eff
            if lib.sg_conv_pack_multi_supported(C.byref(d), C.c_void_p(src.data_ptr())):
                jobs.append((lay, key, d, src, buf))
    for i in range(0, len(jobs), 32):
        chunk = jobs[i:i + 32]
        k = len(chunk)
        descs = (C.POINTER(_abi.ConvDesc) * k)(*[C.pointer(j[2]) for j in chunk])
        srcs = (C.c_void_p * k)(*[j[3].data_ptr() for j in chunk])
        dsts = (C.c_void_p * k)(*[j[4].data_ptr() for j in chunk])
        _abi.call.sg_conv_pack_weights_multi(rt.ctx, k, descs, srcs, dsts)
        for lay, key, d, src, buf in chunk:
            lay._packed[key] = (lay.store.version, buf, d)
    return len(jobs)


class ConvTransposeLayer:
    """tf.keras.layers.Conv2DTranspose(filters, (k,k), strides=(sy,sx), padding='same') -- kernel (kh,kw,Cout,Cin).
    Forward is phase-decomposed (no zero-stuffed MACs): one launch per output phase, each a small stride-1 conv
    with strided output placement.  Reference: resnet_ops.py:57 (3x3) and :69 (1x1 shortcut)."""

    def __init__(self, store: ParamStore, name: str, k: int, ci: int, co: int, strides: Tuple[int, int], init=init_orthogonal):
        self.k, self.ci, self.co = k, ci, co
        self.sy, self.sx = strides
        self.w: Variable = store.add(name + ".w", (k, k, co, ci), init)
        self.b: Variable = store.add(name + ".b", (co,), init_zeros)
        self.store = store
        self.phases = ops.convT_phases(k, self.sy, self.sx)
        self._descs: Dict[tuple, object] = {}
        self._packed: Dict[tuple, Tuple[int, torch.Tensor]] = {}

    def _pack(self, rt, key, d):
        if not ops.tc_ok(rt, d):
            return None
        key = (key, d.in_dt)
        ent = self._packed.get(key)
        if ent is None or ent[0] != self.store.version:
            buf = ops.pack_weights(rt, d, self.w.eff, ent[1] if ent is not None else None)
            self._packed[key] = (self.store.version, buf, d)
            return buf
        return ent[1]

    def forward(self, rt: Runtime, x: torch.Tensor, out=None, accumulate: bool = False, bias="own") -> torch.Tensor:
        """out (fp32) [n, h*sy, w*sx, co].  With accumulate=True the phase results are added into `out` (used for the
        1x1 shortcut, whose bias is folded into the main branch by the caller)."""
        n, h, w, _ = x.shape
        if out is None:
            out = rt.empty((n, h * self.sy, w * self.sx, self.co), SG_F32)
        b = self.b.data if isinstance(bias, str) else bias
        full_cover = len(self.phases) == self.sy * self.sx
        assert accumulate or full_cover, "a transposed conv whose phases do not tile the output must accumulate"
        descs = []
        for (py, px) in self.phases:
            key = ("ph", py, px, n, h, w, dt_of(x), int(accumulate))
            d = self._descs.get(key)
            if d is None:
                d = ops.desc_convT_phase(n, h, w, self.ci, self.co, self.k, self.sy, self.sx, py, px, dt_of(x), SG_F32, 0,
                                         int(accumulate))
                self._descs[key] = d
            descs.append(d)
        if len(descs) > 1 and all(ops.direct_ok(rt, d) for d in descs):
            ops.conv_run_phases(rt, descs, x, self.w.mirror(rt), b, out)       # every phase in ONE launch
            return out
        for (py, px), d in zip(self.phases, descs):
            if ops.direct_ok(rt, d):
                ops.conv_run(rt, d, x, self.w.eff, None, b, None, out, w_mirror=self.w.mirror(rt))
            else:
                ops.conv_run(rt, d, x, self.w.eff, self._pack(rt, ("ph", py, px), d), b, None, out)
        return out

    def _dgrad_desc(self, n, h, w, in_dt, out_dt, accumulate, mask_dt=SG_F32):
        key = ("dg", n, h, w, in_dt, out_dt, accumulate, mask_dt)
        d = self._descs.get(key)
        if d is None:
            d = ops.desc_convT_dgrad(n, h, w, self.ci, self.co, self.k, self.sy, self.sx, in_dt, out_dt, accumulate, mask_dt)
            self._descs[key] = d
        return d

    def dgrad(self, rt: Runtime, dout: torch.Tensor, out_dt: int = SG_F32, out=None, accumulate: bool = False) -> torch.Tensor:
        n, h2, w2, _ = dout.shape
        h, w = h2 // self.sy, w2 // self.sx
        odt = out_dt if out is None else dt_of(out)
        d = self._dgrad_desc(n, h, w, dt_of(dout), odt, int(accumulate))
        if out is None:
            out = rt.empty((n, h, w, self.ci), out_dt)
        if ops.direct_ok(rt, d):
            ops.conv_run(rt, d, dout, self.w.eff, None, None, None, out, w_mirror=self.w.mirror(rt))
        else:
            ops.conv_run(rt, d, dout, self.w.eff, self._pack(rt, "dg", d), None, None, out)
        return out

    def wgrad(self, rt: Runtime, x: torch.Tensor, dout: torch.Tensor, bias_grad: bool = True) -> None:
        """x = layer input [n,h,w,ci], dout = gradient of the output [n,h*sy,w*sx,co] (same dtype as x on the TC path)."""
        n, h, w, _ = x.shape
        d = self._dgrad_desc(n, h, w, dt_of(dout), dt_of(x), 0)
        ops.conv_wgrad(rt, d, dout, x, self.w.grad)
        if bias_grad:
            ops.colsum_into(rt, dout, self.co, self.b.grad, accumulate=1)


class DenseLayer:
    """tf.keras.layers.Dense(units, use_bias) -- kernel (in, out).  resnet_ops.py:18,24; net_architecture.py:55,251,342."""

    def __init__(self, store: ParamStore, name: str, cin: int, cout: int, use_bias: bool = False, init=init_orthogonal):
        self.cin, self.cout = cin, cout
        self.w: Variable = store.add(name + ".w", (cin, cout), init)
        self.b: Optional[Variable] = store.add(name + ".b", (cout,), init_zeros) if use_bias else None

    def forward(self, rt, x, rows: int, ldx: Optional[int] = None) -> torch.Tensor:
        return ops.gemm(rt, x, self.w.eff, rows, self.cout, self.cin, lda=ldx,
                        bias=self.b.data if self.b is not None else None)

    def backward(self, rt, x, dy, rows: int, ldx: Optional[int] = None, want_dx: bool = True, wgrad: bool = True):
        if wgrad:
            ops.gemm(rt, x, dy, self.cin, self.cout, rows, trans_a=True, lda=ldx if ldx is not None else self.cin,
                     out=self.w.grad, accumulate=1)
            if self.b is not None:
                ops.colsum_into(rt, dy, self.cout, self.b.grad, accumulate=1)
        if want_dx:
            return ops.gemm(rt, dy, self.w.eff, rows, self.cin, self.cout, trans_b=True)
        return None


class BatchNormState:
    """Moving statistics (+ optional gamma/beta) of a Keras BatchNormalization layer."""

    def __init__(self, store: ParamStore, name: str, c: int, affine: bool):
        self.c = c
        self.gamma = store.add(name + ".gamma", (c,), init_ones) if affine else None
        self.beta = store.add(name + ".beta", (c,), init_zeros) if affine else None
        self.moving_mean = store.add(name + ".moving_mean", (c,), init_zeros, trainable=False)
        self.moving_var = store.add(name + ".moving_var", (c,), init_ones, trainable=False)


def batch_stats(rt: Runtime, x: torch.Tensor, bn: BatchNormState, update_moving: bool = True):
    """Training-mode statistics over the GLOBAL batch (sync-BN).  With the NVLink peer-memory path up, the second stage
    of the reduction, the cross-replica exchange and the finalisation are ONE launch (sg_bn_finalize_peer); otherwise the
    raw sums are all-reduced with NCCL between sg_bn_stats and sg_bn_finalize."""
    c = x.shape[-1]
    count = x.numel() // c
    mm = bn.moving_mean.data if update_moving else None
    mv = bn.moving_var.data if update_moving else None
    if rt.diag_local_small:                     # timing diagnostics only (WRONG statistics on > 1 replica): no exchange
        sums = ops.bn_stats(rt, x)
        mean, rstd = ops.bn_finalize(rt, sums, count, c, mm, mv)
        return mean, rstd, count
    if rt.world_size > 1 and rt.peer is not None:
        return ops.bn_stats_finalize_peer(rt, x, count * rt.world_size, c, mm, mv) + (count * rt.world_size,)
    # (on a single replica the one-block fused launch is slower than the wide stage-2 + finalize pair: 260 vs 150 us per
    #  step over G's 7 BN layers, profiles/r01_launches_step.csv -- it only pays when it replaces a NCCL call)
    sums = ops.bn_stats(rt, x)
    if rt.world_size > 1:
        rt.allreduce_(sums)
        count *= rt.world_size
    mean, rstd = ops.bn_finalize(rt, sums, count, c, mm, mv)
    return mean, rstd, count
