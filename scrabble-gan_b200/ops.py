"""Functional wrappers over the libsgan C ABI operating on torch CUDA tensors (memory only), plus the
sg_conv_desc builders that express Conv2D / its dgrad / Conv2DTranspose phases / its dgrad with TensorFlow's
SAME / VALID padding rules (SURVEY.md section 8c items 1-2).

Nothing in this file computes on the host or with torch ops: every function is one (or a few) libsgan launches."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _abi
from ._abi import SG_BF16, SG_F32, ConvDesc, call
from .runtime import Runtime, dt_of

_V = C.c_void_p


def _p(t) -> _V:
    return _V(None if t is None else t.data_ptr())


# ----------------------------------------------------------------------------------------------------
# descriptor builders
# ----------------------------------------------------------------------------------------------------
def _same_pad_before(k: int, s: int = 1) -> int:
    """TF SAME: pad_total = max(k - s, 0) when the size is a multiple of s; pad_before = total // 2."""
    return max(k - s, 0) // 2


def _fill_taps(d: ConvDesc, taps) -> None:
    assert 1 <= len(taps) <= _abi.SG_MAX_TAPS, "too many taps"
    d.ntaps = len(taps)
    for i, (dy, dx, off) in enumerate(taps):
        d.tap_dy[i], d.tap_dx[i], d.tap_w_off[i] = dy, dx, off


def desc_conv_fwd(n, h, w, ci, co, kh, kw, padding="same", in_dt=SG_F32, out_dt=SG_F32, relu=0, accumulate=0,
                  mask_dt=SG_F32) -> ConvDesc:
    """tf.keras.layers.Conv2D stride 1, kernel HWIO."""
    d = ConvDesc()
    if padding == "same":
        pt, pl, ho, wo = _same_pad_before(kh), _same_pad_before(kw), h, w
    else:
        pt, pl, ho, wo = 0, 0, h - kh + 1, w - kw + 1
    d.n, d.in_h, d.in_w, d.c_in = n, h, w, ci
    d.out_h, d.out_w, d.c_out = ho, wo, co
    d.grid_h, d.grid_w = ho, wo
    d.in_sy = d.in_sx = d.out_sy = d.out_sx = 1
    d.out_py = d.out_px = 0
    _fill_taps(d, [(a - pt, b - pl, (a * kw + b) * ci * co) for a in range(kh) for b in range(kw)])
    d.w_ci_stride, d.w_co_stride = co, 1
    d.in_dt, d.out_dt, d.relu, d.accumulate, d.mask_dt = in_dt, out_dt, relu, accumulate, mask_dt
    return d


def desc_conv_dgrad(n, h, w, ci, co, kh, kw, padding="same", in_dt=SG_F32, out_dt=SG_F32, accumulate=0,
                    mask_dt=SG_F32) -> ConvDesc:
    """Input gradient of the Conv2D above: `in` = dy [n,ho,wo,co], `out` = dx [n,h,w,ci]; same HWIO master weights."""
    d = ConvDesc()
    if padding == "same":
        pt, pl, ho, wo = _same_pad_before(kh), _same_pad_before(kw), h, w
    else:
        pt, pl, ho, wo = 0, 0, h - kh + 1, w - kw + 1
    d.n, d.in_h, d.in_w, d.c_in = n, ho, wo, co
    d.out_h, d.out_w, d.c_out = h, w, ci
    d.grid_h, d.grid_w = h, w
    d.in_sy = d.in_sx = d.out_sy = d.out_sx = 1
    d.out_py = d.out_px = 0
    _fill_taps(d, [(pt - a, pl - b, (a * kw + b) * ci * co) for a in range(kh) for b in range(kw)])
    d.w_ci_stride, d.w_co_stride = 1, co          # desc "ci" runs over the conv's co and vice versa
    d.in_dt, d.out_dt, d.relu, d.accumulate, d.mask_dt = in_dt, out_dt, 0, accumulate, mask_dt
    return d


def convT_phases(k: int, sy: int, sx: int):
    """Output phases (py, px) of a k x k Conv2DTranspose with strides (sy, sx) that receive at least one tap."""
    pby, pbx = _same_pad_before(k, sy), _same_pad_before(k, sx)
    out = []
    for py in range(sy):
        for px in range(sx):
            ta = [a for a in range(k) if (py + pby - a) % sy == 0]
            tb = [b for b in range(k) if (px + pbx - b) % sx == 0]
            if ta and tb:
                out.append((py, px))
    return out


def desc_convT_phase(n, h, w, ci, co, k, sy, sx, py, px, in_dt=SG_F32, out_dt=SG_F32, relu=0, accumulate=0) -> ConvDesc:
    """One output phase of tf.keras.layers.Conv2DTranspose(k, strides=(sy,sx), 'same'), kernel (kh,kw,Cout,Cin):
    out[n, oy*sy+py, ox*sx+px, :] = sum over taps a == py+pb (mod sy) of in[n, oy + (py+pb-a)/sy, ...] W[a,b]."""
    d = ConvDesc()
    pby, pbx = _same_pad_before(k, sy), _same_pad_before(k, sx)
    d.n, d.in_h, d.in_w, d.c_in = n, h, w, ci
    d.out_h, d.out_w, d.c_out = h * sy, w * sx, co
    d.grid_h, d.grid_w = h, w
    d.in_sy = d.in_sx = 1
    d.out_sy, d.out_sx, d.out_py, d.out_px = sy, sx, py, px
    taps = []
    for a in range(k):
        if (py + pby - a) % sy:
            continue
        for b in range(k):
            if (px + pbx - b) % sx:
                continue
            taps.append(((py + pby - a) // sy, (px + pbx - b) // sx, (a * k + b) * co * ci))
    _fill_taps(d, taps)
    d.w_ci_stride, d.w_co_stride = 1, ci
    d.in_dt, d.out_dt, d.relu, d.accumulate, d.mask_dt = in_dt, out_dt, relu, accumulate, SG_F32
    return d


def desc_convT_dgrad(n, h, w, ci, co, k, sy, sx, in_dt=SG_F32, out_dt=SG_F32, accumulate=0, mask_dt=SG_F32) -> ConvDesc:
    """Input gradient of the Conv2DTranspose: `in` = dout [n,h*sy,w*sx,co] sampled with stride, `out` = dx [n,h,w,ci].
    The filter gradient of the transposed conv is sg_conv_wgrad on THIS descriptor with (in=dout, dy=layer input)."""
    d = ConvDesc()
    pby, pbx = _same_pad_before(k, sy), _same_pad_before(k, sx)
    d.n, d.in_h, d.in_w, d.c_in = n, h * sy, w * sx, co
    d.out_h, d.out_w, d.c_out = h, w, ci
    d.grid_h, d.grid_w = h, w
    d.in_sy, d.in_sx = sy, sx
    d.out_sy = d.out_sx = 1
    d.out_py = d.out_px = 0
    _fill_taps(d, [(a - pby, b - pbx, (a * k + b) * co * ci) for a in range(k) for b in range(k)])
    d.w_ci_stride, d.w_co_stride = ci, 1
    d.in_dt, d.out_dt, d.relu, d.accumulate, d.mask_dt = in_dt, out_dt, 0, accumulate, mask_dt
    return d


# ----------------------------------------------------------------------------------------------------
# convolution launches
# ----------------------------------------------------------------------------------------------------
def tc_ok(rt: Runtime, d: ConvDesc) -> bool:
    return bool(rt.use_tc and _abi.load().sg_conv_tc_supported(C.byref(d)))


def pack_weights(rt: Runtime, d: ConvDesc, w_master: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    n = d.c_out * d.ntaps * d.c_in
    if out is None:
        out = rt.empty((n,), d.in_dt)
    call.sg_conv_pack_weights(rt.ctx, C.byref(d), _p(w_master), _p(out))
    return out


def direct_ok(rt: Runtime, d: ConvDesc, force: bool = False) -> bool:
    """True when the tensor-core launch should read the filter in place from the store's bf16 mirror (no packing pass).
    By default only roles for which the master layout is already K-major (dgrads of Conv2D, phases of Conv2DTranspose):
    reading an HWIO filter in place makes it an N-major UMMA operand, which measured ~20% slower on the big forward
    convs than the packed K-major copy (profiles/), more than the packing pass costs."""
    if not (rt.mode == "bf16" and _abi.load().sg_conv_tc_direct_supported(C.byref(d))):
        return False
    return force or d.w_ci_stride == 1


class _Traced:
    """Diagnostics (tools/trace_step.py): with rt.trace a list, every convolution launch is bracketed by CUDA events and
    recorded as (role, desc summary, start event, end event).  rt.trace is None in normal operation (one attribute test)."""

    def __init__(self, rt, role, d, d2=None):
        self.rt, self.role, self.d, self.d2 = rt, role, d, d2

    def __enter__(self):
        if self.rt.trace is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record(torch.cuda.current_stream(self.rt.device))
        return self

    def __exit__(self, *exc):
        if self.rt.trace is not None:
            self.e1.record(torch.cuda.current_stream(self.rt.device))
            d = self.d
            k = d.ntaps * d.c_in + (self.d2.ntaps * self.d2.c_in if self.d2 is not None else 0)
            self.rt.trace.append((self.role, dict(n=d.n, in_hw=(d.in_h, d.in_w), grid_hw=(d.grid_h, d.grid_w), ci=d.c_in, co=d.c_out, taps=d.ntaps,
                                                  m=d.n * d.grid_h * d.grid_w, k=k, stride=(d.out_sy, d.out_sx), in_stride=(d.in_sy, d.in_sx),
                                                  relu=d.relu, acc=d.accumulate), self.e0, self.e1))
        return False


def conv_run(rt: Runtime, d: ConvDesc, x, w_master, w_packed, bias, mask, out, w_mirror=None) -> None:
    """Launch the conv described by d on the tensor-core path when possible, else the fp32 direct path.  `w_mirror`:
    bf16 mirror of w_master (same layout) for the pack-free tensor-core launch."""
    if rt.trace is not None:
        role = "tc_direct" if w_mirror is not None else ("tc" if (w_packed is not None and tc_ok(rt, d)) else "simt")
        with _Traced(rt, role, d):
            _conv_run(rt, d, x, w_master, w_packed, bias, mask, out, w_mirror)
        return
    _conv_run(rt, d, x, w_master, w_packed, bias, mask, out, w_mirror)


def _conv_run(rt: Runtime, d: ConvDesc, x, w_master, w_packed, bias, mask, out, w_mirror=None) -> None:
    if w_mirror is not None:
        call.sg_conv_fwd_tc_direct(rt.ctx, C.byref(d), _p(x), _p(w_mirror), _p(bias), _p(mask), _p(out))
    elif w_packed is not None and tc_ok(rt, d):
        call.sg_conv_fwd_tc(rt.ctx, C.byref(d), _p(x), _p(w_packed), _p(bias), _p(mask), _p(out))
    else:
        call.sg_conv_fwd_simt(rt.ctx, C.byref(d), _p(x), _p(w_master), _p(bias), _p(mask), _p(out))


def conv_run_rank1(rt: Runtime, d: ConvDesc, x, w_packed, bias, mask, out, r1_x, r1_w) -> None:
    """Tensor-core conv with the rank-1 epilogue term out[p, c] += r1_x[p] * r1_w[c] (a 1x1 conv of a one-channel tensor)."""
    with _Traced(rt, "tc_rank1", d):
        call.sg_conv_fwd_tc_rank1(rt.ctx, C.byref(d), _p(x), _p(w_packed), _p(bias), _p(mask), _p(out), _p(r1_x), _p(r1_w))


def conv_run_phases(rt: Runtime, descs, x, w_mirror, bias, out) -> None:
    """All output phases of a transposed conv in ONE tensor-core launch (filter read in place from the bf16 mirror)."""
    k = len(descs)
    arr = (C.POINTER(ConvDesc) * k)(*[C.pointer(d) for d in descs])
    if rt.trace is not None:
        import copy
        dsum = copy.copy(descs[0])
        d2 = None
        with _Traced(rt, "tc_phases", dsum, d2) as tr:
            call.sg_conv_fwd_tc_phases(rt.ctx, k, arr, _p(x), _p(w_mirror), _p(bias), _p(out))
        role, info, e0, e1 = rt.trace[-1]
        info["taps"] = sum(d.ntaps for d in descs)
        info["k"] = info["taps"] * descs[0].c_in
        return
    call.sg_conv_fwd_tc_phases(rt.ctx, k, arr, _p(x), _p(w_mirror), _p(bias), _p(out))


def conv_run_dual(rt: Runtime, d: ConvDesc, x, w_packed, d2: ConvDesc, x2, w_packed2, bias, mask, out) -> None:
    """Main conv + 1x1 shortcut conv accumulated in ONE tensor-core launch (both filters packed)."""
    with _Traced(rt, "tc_dual", d, d2):
        call.sg_conv_fwd_tc_dual(rt.ctx, C.byref(d), _p(x), _p(w_packed), C.byref(d2), _p(x2), _p(w_packed2), _p(bias), _p(mask), _p(out))


def conv_wgrad(rt: Runtime, d: ConvDesc, x, dy, dw_master, force_simt: bool = False, db=None, db2=None, force_bias: bool = False) -> bool:
    if rt.trace is not None:
        with _Traced(rt, "wgrad", d):
            return _conv_wgrad(rt, d, x, dy, dw_master, force_simt, db, db2, force_bias)
    return _conv_wgrad(rt, d, x, dy, dw_master, force_simt, db, db2, force_bias)


def _conv_wgrad(rt: Runtime, d: ConvDesc, x, dy, dw_master, force_simt: bool = False, db=None, db2=None, force_bias: bool = False) -> bool:
    """dw_master += filter gradient of the conv described by d: on the tensor cores whenever the layer is eligible and both
    operands have the mode's operand dtype (bf16, or fp32 read as tf32 in "tf32" mode); the FFMA kernel serves the edge
    layers (Cin = 1 / Cout = 1) and the exact "fp32" mode -- by rule, not as a silent fallback.
    db (and db2): bias gradient(s) to accumulate the column sums of dy into IN THE SAME LAUNCH; returns True when that was
    done (tensor-core path of a plain Conv2D whose extra bias units fit into the idle slots of the launch's last wave --
    sg_conv_wgrad_tc_bias_fits; force_bias skips that test), False when the caller still has to sum dy itself."""
    tc_dt = SG_BF16 if rt.mode == "bf16" else (SG_F32 if rt.mode == "tf32" else None)
    if not force_simt and tc_dt is not None and d.in_dt == tc_dt and d.out_dt == tc_dt and tc_ok(rt, d):
        if db is not None and d.out_sy == 1 and d.out_sx == 1 and d.grid_h == d.out_h and d.grid_w == d.out_w and \
                (force_bias or _abi.load().sg_conv_wgrad_tc_bias_fits(rt.ctx, C.byref(d))):
            call.sg_conv_wgrad_tc_bias(rt.ctx, C.byref(d), _p(x), _p(dy), _p(dw_master), _p(db), _p(db2))
            return True
        call.sg_conv_wgrad_tc(rt.ctx, C.byref(d), _p(x), _p(dy), _p(dw_master), _V(None), 0)
    else:
        if rt.use_tc and tc_ok(rt, d) and not force_simt and d.in_dt != d.out_dt:
            raise _abi.SganError("conv_wgrad: tensor-core layer with mixed operand dtypes (in {}, dy {}): the producer must write the "
                                 "operand dtype".format(d.in_dt, d.out_dt))
        call.sg_conv_wgrad_simt(rt.ctx, C.byref(d), _p(x), _p(dy), _p(dw_master))
    return False


# ----------------------------------------------------------------------------------------------------
# element-wise, pooling
# ----------------------------------------------------------------------------------------------------
def act_prep(rt, x, want_relu=True, want_copy=False, out_dt=None):
    out_dt = rt.op_dt if out_dt is None else out_dt
    r = rt.empty(x.shape, out_dt) if want_relu else None
    c = rt.empty(x.shape, out_dt) if want_copy else None
    call.sg_act_prep(rt.ctx, _p(x), x.numel(), _p(r), _p(c), out_dt)
    return r, c


def cast(rt, x, out_dt):
    if dt_of(x) == out_dt:
        return x
    out = rt.empty(x.shape, out_dt)
    call.sg_cast(rt.ctx, _p(x), _p(out), out_dt, x.numel())
    return out


def mask_mul(rt, dy, act, out_dt=SG_F32, out=None, accumulate=0):
    if out is None:
        out = rt.empty(dy.shape, out_dt)
    call.sg_mask_mul(rt.ctx, _p(dy), _p(act), dt_of(act), _p(out), dt_of(out), dy.numel(), accumulate)
    return out


def axpby(rt, a, x, b=0.0, y=None, out=None):
    if out is None:
        out = rt.empty(x.shape, SG_F32)
    call.sg_axpby(rt.ctx, float(a), _p(x), float(b), _p(y), _p(out), x.numel())
    return out


def scale_add(rt, sigma, a, x=None, out=None):
    if out is None:
        out = rt.empty(a.shape, SG_F32)
    call.sg_scale_add(rt.ctx, _p(sigma), _p(a), _p(x), _p(out), a.numel())
    return out


def tanh_fwd(rt, x, out=None):
    y = rt.empty(x.shape, SG_F32) if out is None else out
    call.sg_tanh_fwd(rt.ctx, _p(x), _p(y), x.numel())
    return y


def tanh_bwd(rt, dy, y):
    dx = rt.empty(y.shape, SG_F32)
    call.sg_tanh_bwd(rt.ctx, _p(dy), _p(y), _p(dx), y.numel())
    return dx


def scale_rows_(rt, x, w):
    rows = w.numel()
    call.sg_scale_rows(rt.ctx, _p(x), _p(w), rows, x.numel() // rows)
    return x


def scale_samples_(rt, x, up, mult: float):
    """In place: x[i] *= up[i] * mult for the samples i of the batch-first tensor x (fp32 or bf16)."""
    n = x.shape[0]
    call.sg_scale_samples(rt.ctx, _p(x), dt_of(x), n, x.numel() // max(n, 1), _p(up), float(mult))
    return x


def dot_into(rt, a, b, out, accumulate=1):
    call.sg_dot(rt.ctx, _p(a), _p(b), a.numel(), _p(out), accumulate)


def colsum_into(rt, x, cols, out, accumulate=1):
    call.sg_colsum(rt.ctx, _p(x), dt_of(x), x.numel() // cols, cols, _p(out), accumulate)


def avgpool2_fwd(rt, x):
    n, h, w, c = x.shape
    out = rt.empty((n, h // 2, w // 2, c), SG_F32)
    call.sg_avgpool2_fwd(rt.ctx, _p(x), n, h, w, c, _p(out))
    return out


def avgpool2_bwd(rt, dout, out_dt):
    n, ho, wo, c = dout.shape
    dx = rt.empty((n, ho * 2, wo * 2, c), out_dt)
    call.sg_avgpool2_bwd(rt.ctx, _p(dout), n, ho * 2, wo * 2, c, _p(dx), out_dt)
    return dx


def maxpool_fwd(rt, x, ph, pw):
    n, h, w, c = x.shape
    out = torch.empty((n, h // ph, w // pw, c), device=x.device, dtype=x.dtype)
    call.sg_maxpool_fwd(rt.ctx, _p(x), dt_of(x), n, h, w, c, ph, pw, _p(out))
    return out


def maxpool_bwd(rt, dout, x, ph, pw, relu_mask, out_dt):
    n, h, w, c = x.shape
    dx = rt.empty(x.shape, out_dt)
    call.sg_maxpool_bwd(rt.ctx, _p(dout), _p(x), dt_of(x), n, h, w, c, ph, pw, int(relu_mask), _p(dx), out_dt)
    return dx


def gap_relu_fwd(rt, x):
    n, h, w, c = x.shape
    out = rt.empty((n, c), SG_F32)
    call.sg_gap_relu_fwd(rt.ctx, _p(x), n, h * w, c, _p(out))
    return out


def gap_relu_bwd(rt, dfeat, x):
    n, h, w, c = x.shape
    dx = rt.empty(x.shape, SG_F32)
    call.sg_gap_relu_bwd(rt.ctx, _p(dfeat), _p(x), n, h * w, c, _p(dx))
    return dx


# ----------------------------------------------------------------------------------------------------
# batch norm
# ----------------------------------------------------------------------------------------------------
def bn_stats(rt, x) -> torch.Tensor:
    """[2C] raw sums (sum x, sum x^2) over all rows of x [.., C]; all-reduced across replicas by the caller."""
    c = x.shape[-1]
    rows = x.numel() // c
    nbytes = _abi.load().sg_bn_stats_scratch_bytes(rows, c)
    scratch = rt.scratch("bn" if rt.ctx is rt._main_ctx else "bn_side", nbytes)      # one scratch per stream: never shared by concurrent kernels
    sums = rt.empty((2 * c,), SG_F32)
    call.sg_bn_stats(rt.ctx, _p(x), rows, c, _p(sums), _p(scratch), nbytes)
    return sums


def bn_stats_finalize_peer(rt, x, count_total, c, moving_mean=None, moving_var=None, eps=1e-3, momentum=0.99, pe=None):
    """sync-BN statistics with the cross-replica exchange fused into the finalisation (needs rt.peer): the wide two-stage sum
    of this replica (sg_bn_stats), then ONE small launch doing NVLink exchange + mean / rstd / moving averages.  (Stage 2
    used to run inside that one-block launch as well: 16 us per layer slower than the wide stage-2 kernel, measured.)"""
    pe = rt.peer if pe is None else pe
    sums = bn_stats(rt, x)
    mean, rstd = rt.empty((c,), SG_F32), rt.empty((c,), SG_F32)
    call.sg_bn_finalize_peer(rt.ctx, _p(sums), 1, c, float(count_total), eps, momentum, _V(None), _p(mean), _p(rstd),
                             _p(moving_mean), _p(moving_var), pe.ptrs, pe.world, pe.rank)
    return mean, rstd


def bn_finalize(rt, sums, count, c, moving_mean=None, moving_var=None, eps=1e-3, momentum=0.99):
    mean, rstd = rt.empty((c,), SG_F32), rt.empty((c,), SG_F32)
    call.sg_bn_finalize(rt.ctx, _p(sums), float(count), c, eps, momentum, _p(mean), _p(rstd), _p(moving_mean), _p(moving_var))
    return mean, rstd


def bn_infer_prepare(rt, moving_mean, moving_var, eps=1e-3):
    c = moving_mean.numel()
    mean, rstd = rt.empty((c,), SG_F32), rt.empty((c,), SG_F32)
    call.sg_bn_infer_prepare(rt.ctx, _p(moving_mean), _p(moving_var), c, eps, _p(mean), _p(rstd))
    return mean, rstd


def bn_apply(rt, x, mean, rstd, gamma, beta, per_sample: bool, relu: bool, out_dt, gb_stride=None):
    """gb_stride: row stride of per-sample gamma / beta (default c; the grouped CBN Dense output has a wider row)."""
    n, c = x.shape[0], x.shape[-1]
    hw = x.numel() // (n * c)
    out = rt.empty(x.shape, out_dt)
    stride = (c if gb_stride is None else gb_stride) if per_sample else 0
    call.sg_bn_apply(rt.ctx, _p(x), n, hw, c, _p(mean), _p(rstd), _p(gamma), _p(beta), stride, int(relu), _p(out), out_dt)
    return out


def bn_bwd_reduce(rt, dy, act, x, mean, rstd):
    n, c = x.shape[0], x.shape[-1]
    hw = x.numel() // (n * c)
    s1, s2 = rt.empty((n, c), SG_F32), rt.empty((n, c), SG_F32)
    call.sg_bn_bwd_reduce(rt.ctx, _p(dy), _p(act), dt_of(act) if act is not None else SG_F32, _p(x), n, hw, c, _p(mean),
                          _p(rstd), _p(s1), _p(s2))
    return s1, s2


def bn_bwd_combine(rt, s1, s2, gamma, per_sample: bool, gb_stride=None):
    n, c = s1.shape
    ab = rt.empty((2 * c,), SG_F32)
    stride = (c if gb_stride is None else gb_stride) if per_sample else 0
    call.sg_bn_bwd_combine(rt.ctx, _p(s1), _p(s2), _p(gamma), stride, n, c, _p(ab))
    return ab


def bn_bwd_apply(rt, dy, act, x, mean, rstd, gamma, per_sample, ab, count, use_batch_terms, mask_by_x, out_dt, out=None,
                 accumulate=0, gb_stride=None):
    n, c = x.shape[0], x.shape[-1]
    hw = x.numel() // (n * c)
    if out is None:
        out = rt.empty(x.shape, out_dt)
    stride = (c if gb_stride is None else gb_stride) if per_sample else 0
    call.sg_bn_bwd_apply(rt.ctx, _p(dy), _p(act), dt_of(act) if act is not None else SG_F32, _p(x), n, hw, c, _p(mean), _p(rstd),
                         _p(gamma), stride, _p(ab), float(count), int(use_batch_terms), int(mask_by_x), _p(out),
                         dt_of(out), accumulate)
    return out


def cbn_dense_fwd(rt, z, z_stride, n, segs, w_base):
    """segs: [(c, z_off, w_off)]: all CBN gamma / beta Dense layers of the generator in ONE launch -> [n, sum c]."""
    k = len(segs)
    total = sum(s[0] for s in segs)
    out = rt.empty((n, total), SG_F32)
    ci = (C.c_int * k)(*[s[0] for s in segs])
    zi = (C.c_int * k)(*[s[1] for s in segs])
    wi = (C.c_longlong * k)(*[s[2] for s in segs])
    call.sg_cbn_dense_fwd(rt.ctx, _p(z), z_stride, n, k, ci, zi, wi, _p(w_base), _p(out))
    return out


def cbn_dense_wgrad(rt, z, z_stride, n, segs, upstream, dw_base):
    """dW of every segment in ONE launch; upstream[i]: [n, c_i] contiguous."""
    k = len(segs)
    ci = (C.c_int * k)(*[s[0] for s in segs])
    zi = (C.c_int * k)(*[s[1] for s in segs])
    wi = (C.c_longlong * k)(*[s[2] for s in segs])
    up = (C.c_void_p * k)(*[u.data_ptr() for u in upstream])
    call.sg_cbn_dense_wgrad(rt.ctx, _p(z), z_stride, n, k, ci, zi, wi, up, _p(dw_base))


# ----------------------------------------------------------------------------------------------------
# dense, filter bank, attention, CTC, losses, optimizers, spectral norm
# ----------------------------------------------------------------------------------------------------
def gemm(rt, a, b, m, n, k, trans_a=False, trans_b=False, lda=None, ldb=None, out=None, ldc=None, bias=None, accumulate=0):
    """out[m,n] (+)= op(a)[m,k] @ op(b)[k,n] + bias; row-major with explicit leading dimensions."""
    if lda is None:
        lda = m if trans_a else k
    if ldb is None:
        ldb = k if trans_b else n
    if out is None:
        out = rt.empty((m, n), SG_F32)
    if ldc is None:
        ldc = n
    call.sg_gemm(rt.ctx, int(trans_a), int(trans_b), m, n, k, _p(a), lda, _p(b), ldb, _p(out), ldc, _p(bias), accumulate)
    return out


def filterbank_fwd(rt, z, z_stride, y, bank):
    b, l = y.shape
    out = rt.empty((b, 4, 4 * l, 512), SG_F32)
    call.sg_filterbank_fwd(rt.ctx, _p(z), z_stride, _p(y), b, l, bank.shape[0], _p(bank), _p(out))
    return out


def filterbank_bwd(rt, dout, z, z_stride, y, bank, dbank, dz0=None, dz_stride=32):
    """dbank is overwritten; dz0[b*dz_stride + j] (j < 32) is written when given."""
    b, l = y.shape
    call.sg_filterbank_bwd(rt.ctx, _p(dout), _p(z), z_stride, _p(y), b, l, bank.shape[0], _p(bank), _p(dbank), _p(dz0),
                           dz_stride)
    return dz0


def _attn_tc(rt, q, kv, dk, dv, tc) -> bool:
    """Tensor-core attention is the speed-mode ("bf16") path; "fp32"/"tf32" modes keep the exact FFMA kernels."""
    if tc is None:
        tc = rt.mode == "bf16"
    return bool(tc and _abi.load().sg_attn_tc_supported(q, kv, dk, dv))


def label_lengths(rt, labels):
    """lens[b] = number of leading labels >= 0 (ragged batches pad the label matrix with -1)."""
    b, l = labels.shape
    lens = torch.empty((b,), device=rt.device, dtype=torch.int32)
    call.sg_label_lengths(rt.ctx, _p(labels), b, l, _p(lens))
    return lens


def mask_width_(rt, x, lens, cols_per_char: int):
    """In place: zero the NHWC tensor x right of column cols_per_char * lens[n] of every image n."""
    n, h, w, c = x.shape
    call.sg_mask_width(rt.ctx, _p(x), dt_of(x), n, h, w, c, _p(lens), cols_per_char)
    return x


def attn_fwd(rt, theta, phi, g, tc=None, kv_w: int = 0, kv_cols=None):
    """kv_cols (int32 [n]) with kv_w = key columns per row: keys in columns >= kv_cols[n] are left out of image n's softmax."""
    n, q, dk = theta.shape
    kv, dv = g.shape[1], g.shape[2]
    o, lse = rt.empty((n, q, dv), SG_F32), rt.empty((n, q), SG_F32)
    if kv_cols is not None:
        fn = call.sg_attn_fwd_tc_masked if _attn_tc(rt, q, kv, dk, dv, tc) else call.sg_attn_fwd_masked
        fn(rt.ctx, _p(theta), _p(phi), _p(g), n, q, kv, dk, dv, kv_w, _p(kv_cols), _p(o), _p(lse))
        return o, lse
    if _attn_tc(rt, q, kv, dk, dv, tc):
        call.sg_attn_fwd_tc(rt.ctx, _p(theta), _p(phi), _p(g), n, q, kv, dk, dv, _p(o), _p(lse))
    else:
        call.sg_attn_fwd(rt.ctx, _p(theta), _p(phi), _p(g), n, q, kv, dk, dv, _p(o), _p(lse))
    return o, lse


def attn_bwd(rt, theta, phi, g, o, lse, d_o, tc=None):
    n, q, dk = theta.shape
    kv, dv = g.shape[1], g.shape[2]
    dtheta, dphi, dg = rt.empty(theta.shape, SG_F32), rt.empty(phi.shape, SG_F32), rt.empty(g.shape, SG_F32)
    if _attn_tc(rt, q, kv, dk, dv, tc):
        scratch = rt.empty((n, q), SG_F32)
        call.sg_attn_bwd_tc(rt.ctx, _p(theta), _p(phi), _p(g), _p(o), _p(lse), _p(d_o), n, q, kv, dk, dv, _p(dtheta), _p(dphi),
                            _p(dg), _p(scratch))
    else:
        call.sg_attn_bwd(rt.ctx, _p(theta), _p(phi), _p(g), _p(o), _p(lse), _p(d_o), n, q, kv, dk, dv, _p(dtheta), _p(dphi), _p(dg))
    return dtheta, dphi, dg


def nonlocal_proj_fwd(rt, x, w_theta, w_phi, w_g):
    """theta [p,8], phi_f [p,8], g_f [p,32] from ONE pass over x [p,64] (arch_ops.py:38-46,55-57)."""
    p = x.numel() // 64
    theta, phi_f, g_f = rt.empty((p, 8)), rt.empty((p, 8)), rt.empty((p, 32))
    call.sg_nonlocal_proj_fwd(rt.ctx, _p(x), p, _p(w_theta), _p(w_phi), _p(w_g), _p(theta), _p(phi_f), _p(g_f))
    return theta, phi_f, g_f


def nonlocal_out_fwd(rt, o, w_o, sigma, x):
    """og = o @ w_o, out = sigma * og + x (arch_ops.py:63-67)."""
    p = x.numel() // 64
    og, out = rt.empty((p, 64)), rt.empty((p, 64))
    call.sg_nonlocal_out_fwd(rt.ctx, _p(o), p, _p(w_o), _p(sigma), _p(x), _p(og), _p(out))
    return og, out


def nonlocal_out_bwd(rt, dout, o, w_o, sigma, dw_o=None):
    p = dout.numel() // 64
    d_o = rt.empty((p, 32))
    call.sg_nonlocal_out_bwd(rt.ctx, _p(dout), _p(o), p, _p(w_o), _p(sigma), _p(d_o), _p(dw_o))
    return d_o


def nonlocal_proj_bwd(rt, x, dtheta, dphi_f, dg_f, w_theta, w_phi, w_g, dx, dw_theta=None, dw_phi=None, dw_g=None):
    """dx += the three input gradients; dw_* += the three filter gradients (one pass over x each)."""
    p = x.numel() // 64
    call.sg_nonlocal_proj_bwd(rt.ctx, _p(x), _p(dtheta), _p(dphi_f), _p(dg_f), p, _p(w_theta), _p(w_phi), _p(w_g), _p(dx),
                              _p(dw_theta), _p(dw_phi), _p(dw_g))
    return dx


def ctc(rt, logits, labels, want_grad=True, input_length=None, label_length=None):
    """K.ctc_batch_cost: per-sample (B,) int32 device tensors input_length / label_length make the batch ragged."""
    b, t, c = logits.shape
    l = labels.shape[1]
    loss = rt.empty((b,), SG_F32)
    grad = rt.empty(logits.shape, SG_F32) if want_grad else None
    if input_length is None and label_length is None:
        call.sg_ctc(rt.ctx, _p(logits), _p(labels), b, t, c, l, _p(loss), _p(grad))
    else:
        il = input_length if input_length is not None else torch.full((b,), t, device=rt.device, dtype=torch.int32)
        ll = label_length if label_length is not None else torch.full((b,), l, device=rt.device, dtype=torch.int32)
        call.sg_ctc_ragged(rt.ctx, _p(logits), _p(labels), b, t, c, l, _p(il), _p(ll), _p(loss), _p(grad))
    return loss, grad


def softmax_rows(rt, x):
    """Softmax over the last dimension of an fp32 tensor (R's Dense activation)."""
    c = x.shape[-1]
    y = rt.empty(x.shape, SG_F32)
    call.sg_softmax_rows(rt.ctx, _p(x), x.numel() // c, c, _p(y))
    return y


def ctc_greedy_decode(rt, probs, input_length=None):
    """K.ctc_decode(greedy=True) on probs (B, T, C): decoded (B, T) int32 padded with -1, decoded_len (B,) int32,
    neg_sum_log (B,) fp32.  input_length: (B,) int32 device tensor or None (all T frames)."""
    b, t, c = probs.shape
    decoded = torch.empty((b, t), device=rt.device, dtype=torch.int32)
    dlen = torch.empty((b,), device=rt.device, dtype=torch.int32)
    score = rt.empty((b,), SG_F32)
    call.sg_ctc_greedy_decode(rt.ctx, _p(probs), b, t, c, _p(input_length), _p(decoded), _p(dlen), _p(score))
    return decoded, dlen, score


def edit_distance(rt, hyp, ref, hyp_length=None, ref_length=None, totals=None):
    """Levenshtein distance (B,) int32 between the rows of hyp (B, Lh) and ref (B, Lr <= 64); without a length tensor a row
    ends at its first negative entry.  totals: int64 (4,) device tensor that is ADDED to (sum dist, sum ref length, exact
    matches, samples)."""
    b = hyp.shape[0]
    dist = torch.empty((b,), device=rt.device, dtype=torch.int32)
    call.sg_edit_distance(rt.ctx, _p(hyp), _p(hyp_length), hyp.shape[1], _p(ref), _p(ref_length), ref.shape[1], b, _p(dist),
                          _p(totals))
    return dist


def random_(rt, out, normal: bool = True, seed: Optional[int] = None):
    """Fill `out` (fp32) with N(0,1) (or U[-1,1)) numbers from the runtime's Philox stream; the stream position lives on the
    device (rt.rng_state), so the launch can be captured in a CUDA graph and still draw fresh numbers on every replay."""
    st = rt.rng_state()
    call.sg_random(rt.ctx, _p(out), out.numel(), rt.rng_seed if seed is None else int(seed), 0, _p(st), int(normal))
    return out


def adam_(rt, w, g, m, v, lr_t, beta1, beta2, eps, mirror=None):
    if mirror is not None:
        call.sg_adam_mirror(rt.ctx, _p(w), _p(g), _p(m), _p(v), _p(mirror), w.numel(), lr_t, beta1, beta2, eps)
    else:
        call.sg_adam(rt.ctx, _p(w), _p(g), _p(m), _p(v), w.numel(), lr_t, beta1, beta2, eps)


def rmsprop_(rt, w, g, ms, lr, rho, eps):
    call.sg_rmsprop(rt.ctx, _p(w), _p(g), _p(ms), w.numel(), lr, rho, eps)


def spectral_norm(rt, w, u, power_iteration=1):
    """arch_ops.py:99-126 with explicit u [cols]; returns (w / sigma, u_hat, sigma)."""
    cols = w.shape[-1]
    rows = w.numel() // cols
    w_out, u_out, sigma = rt.empty(w.shape, SG_F32), rt.empty((cols,), SG_F32), rt.empty((1,), SG_F32)
    scratch = rt.empty((rows + cols + 4,), SG_F32)
    call.sg_spectral_norm(rt.ctx, _p(w), rows, cols, _p(u), power_iteration, _p(w_out), _p(u_out), _p(sigma), _p(scratch))
    return w_out, u_out, sigma
