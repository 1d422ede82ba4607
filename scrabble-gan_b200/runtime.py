"""Per-process runtime: one sg_ctx bound to one GPU and torch's current stream.

PyTorch is used here for plumbing only: device memory (torch.empty), streams and torch.distributed (NCCL).
All arithmetic is done by libsgan kernels.  Precision modes:
    "bf16"  conv operands bf16, tcgen05 kind::f16, fp32 accumulate            (speed mode, 1e-2 parity)
    "tf32"  conv operands fp32 read as tf32 by tcgen05 kind::tf32             (fp32 storage, ~1e-3 parity)
    "fp32"  exact fp32 FFMA direct convolutions (no tensor cores)            (parity/debug mode)
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

from . import _abi
from ._abi import SG_BF16, SG_F32, call

_MODES = ("bf16", "tf32", "fp32")


class Runtime:
    def __init__(self, device: Optional[int] = None, mode: Optional[str] = None):
        if not torch.cuda.is_available():
            raise _abi.SganError("no CUDA device visible: scrabble-gan_b200 has no CPU path")
        _abi.load()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", torch.cuda.current_device()))
        mode = mode or os.environ.get("SGAN_MODE", "bf16")
        if mode not in _MODES:
            raise ValueError("mode must be one of {}".format(_MODES))
        self.device_index = device
        torch.cuda.set_device(device)
        self.device = torch.device("cuda", device)
        self.stream = torch.cuda.current_stream(self.device)
        handle = C.c_void_p()
        call.sg_ctx_create(device, C.c_void_p(self.stream.cuda_stream), C.byref(handle))
        self.ctx = handle
        self._main_ctx = handle
        # second stream + context for work that is independent of the main stream's (the recogniser's passes next to the
        # discriminator's inside a train step): created on first use by branch()
        self.side_stream = None
        self._side_ctx = None
        self.num_sms = torch.cuda.get_device_properties(device).multi_processor_count
        self.set_mode(mode)
        # data-parallel state (see dp.py)
        self.world_size = 1
        self.rank = 0
        self.process_group = None
        # timing diagnostics of the data-parallel step (they make its results WRONG): skip the small exchanges / G's bucket
        self.diag_local_small = os.environ.get("SGAN_DIAG_LOCAL_SMALL", "0") == "1"
        self.diag_skip_g_bucket = os.environ.get("SGAN_DIAG_SKIP_G_BUCKET", "0") == "1"
        self.peer = None            # dp.PeerExchange when the NVLink peer-memory path is up
        self.peer_comm = None       # a second one: barrier flags of the communication stream (bucket all-reduce)
        self._comm = None           # (stream, context) of the communication stream
        self.replayed_launches = 0  # kernels executed through CUDA-graph replays (they bypass the C ABI's launch counter)
        self._scratch = {}
        self.rng_seed = int(os.environ.get("SGAN_SEED", "1234")) + 7919 * int(os.environ.get("RANK", "0"))
        self._rng_state = None      # device-resident Philox stream position (uint64[1])

    # ---- precision mode -----------------------------------------------------------------------------
    def set_mode(self, mode: str) -> None:
        if mode not in _MODES:
            raise ValueError("mode must be one of {}".format(_MODES))
        self.mode = mode
        self.use_tc = mode in ("bf16", "tf32")
        self.op_dt = SG_BF16 if mode == "bf16" else SG_F32
        self.op_torch = torch.bfloat16 if mode == "bf16" else torch.float32
        self.trace = None                       # diagnostics: a list makes ops.conv_* record (role, shape, events) per launch
        for c in (self._main_ctx, self._side_ctx):
            if c is not None:
                call.sg_ctx_set_speed_mode(c, int(mode == "bf16"))

    # ---- memory helpers (torch = allocator only) ------------------------------------------------------
    def empty(self, shape, dt: int = SG_F32) -> torch.Tensor:
        return torch.empty(shape, device=self.device, dtype=torch.float32 if dt == SG_F32 else torch.bfloat16)

    def empty_op(self, shape) -> torch.Tensor:
        return torch.empty(shape, device=self.device, dtype=self.op_torch)

    def zeros(self, shape, dtype=torch.float32) -> torch.Tensor:
        return torch.zeros(shape, device=self.device, dtype=dtype)

    def scratch(self, key: str, nbytes: int) -> torch.Tensor:
        t = self._scratch.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(max(nbytes, 1), device=self.device, dtype=torch.uint8)
            self._scratch[key] = t
        return t

    def rng_state(self) -> torch.Tensor:
        if self._rng_state is None:
            self._rng_state = torch.zeros(1, device=self.device, dtype=torch.int64)
        return self._rng_state

    def manual_seed(self, seed: int) -> None:
        self.rng_seed = int(seed)
        self.rng_state().zero_()

    # ---- misc ---------------------------------------------------------------------------------------
    def sync(self) -> None:
        call.sg_ctx_sync(self.ctx)

    def launch_count(self) -> int:
        """libsgan kernels launched so far: direct launches through the C ABI plus the kernel nodes of replayed graphs."""
        n = int(_abi.load().sg_ctx_launch_count(self._main_ctx))
        if self._side_ctx is not None:
            n += int(_abi.load().sg_ctx_launch_count(self._side_ctx))
        if self._comm is not None:
            n += int(_abi.load().sg_ctx_launch_count(self._comm[1]))
        return n + self.replayed_launches

    def use_current_stream(self) -> None:
        self.stream = torch.cuda.current_stream(self.device)
        call.sg_ctx_set_stream(self._main_ctx, C.c_void_p(self.stream.cuda_stream))

    def close(self) -> None:
        """Release the libsgan contexts (each owns a 48 MB device workspace).  The runtime must not be used afterwards."""
        torch.cuda.synchronize(self.device)
        for h in (self._main_ctx, self._side_ctx, self._comm[1] if self._comm is not None else None):
            if h is not None:
                _abi.load().sg_ctx_destroy(h)
        self._main_ctx = self._side_ctx = self.ctx = None
        self._comm = None

    def comm_stream_ctx(self):
        """The communication stream and its libsgan context (created on first use): gradient-bucket all-reduces run there."""
        if self._comm is None:
            st = torch.cuda.Stream(device=self.device)
            handle = C.c_void_p()
            call.sg_ctx_create(self.device_index, C.c_void_p(st.cuda_stream), C.byref(handle))
            self._comm = (st, handle)
        return self._comm

    def branch(self) -> "Branch":
        """Fork a branch of independent work onto the side stream:

            br = rt.branch()          # the side stream waits for everything enqueued on the main stream so far
            with br: ...              # launches (and allocations) inside go to the side stream / side context
            ...                       # main-stream work enqueued here runs concurrently with the branch
            br.join()                 # the main stream waits for the branch

        The side context owns its own workspace (deterministic-reduction scratch, tickets), so kernels of the two streams
        never share one."""
        return Branch(self)


    # ---- data parallel (sum all-reduce of small statistic vectors and of gradient buckets) -------------
    def allreduce_(self, t: torch.Tensor) -> torch.Tensor:
        if self.world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.process_group)
        return t

    def allreduce_small_(self, t: torch.Tensor) -> torch.Tensor:
        """SUM all-reduce of a SMALL fp32 / fp64 vector (BN statistics, loss sums): one-shot exchange over NVLink peer
        memory on the compute stream (csrc/peer.cu) when available, NCCL otherwise."""
        if self.world_size <= 1 or self.diag_local_small:
            return t
        pe = self.peer
        if pe is not None and t.is_contiguous() and t.dtype in (torch.float32, torch.float64) and \
                t.numel() * t.element_size() <= self._peer_max():
            call.sg_peer_allreduce_sum(self.ctx, C.c_void_p(t.data_ptr()), t.numel(), int(t.dtype == torch.float64), pe.ptrs,
                                       pe.world, pe.rank)
            return t
        return self.allreduce_(t)

    def _peer_max(self) -> int:
        if not hasattr(self, "_peer_max_bytes"):
            self._peer_max_bytes = int(_abi.load().sg_peer_max_payload_bytes())
        return self._peer_max_bytes

    def allreduce_async_(self, t: torch.Tensor, store=None, exposed: bool = False):
        """Start a SUM all-reduce of `t` on NCCL's own stream (ordered after everything already enqueued on the compute
        stream) and return a handle; compute enqueued afterwards overlaps with the transfer.  `wait()` orders the compute
        stream after the collective.  Returns None on a single replica."""
        if self.world_size <= 1:
            return None
        import torch.distributed as dist
        if store is not None:
            from . import dp
            h = dp.bucket_allreduce_async(self, store, exposed)      # copy engines over NVLink peer memory: no SMs taken from the step
            if h is not None:
                return h
            t = store.g
        if os.environ.get("SGAN_DP_SYNC_ALLREDUCE", "0") == "1":      # diagnostic: no overlap with the backward passes
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.process_group)
            return None
        return dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.process_group, async_op=True)


class Branch:
    def __init__(self, rt: Runtime):
        self.rt = rt
        self._ctxmgr = None
        self._done = None               # event recorded on the side stream at the end of the last `with` block of this branch
        if rt.side_stream is None:
            rt.side_stream = torch.cuda.Stream(device=rt.device)
            handle = C.c_void_p()
            call.sg_ctx_create(rt.device_index, C.c_void_p(rt.side_stream.cuda_stream), C.byref(handle))
            rt._side_ctx = handle
            call.sg_ctx_set_speed_mode(handle, int(rt.mode == "bf16"))
        self.main = torch.cuda.current_stream(rt.device)
        rt.side_stream.wait_stream(self.main)

    def __enter__(self):
        self.rt.ctx = self.rt._side_ctx
        self._ctxmgr = torch.cuda.stream(self.rt.side_stream)
        self._ctxmgr.__enter__()
        return self

    def __exit__(self, *exc):
        self._done = torch.cuda.Event()
        self._done.record(self.rt.side_stream)
        self._ctxmgr.__exit__(*exc)
        self.rt.ctx = self.rt._main_ctx
        return False

    def join(self) -> None:
        """The current stream waits for what THIS branch enqueued (its `with` blocks) -- not for work other branches put on
        the side stream afterwards; a branch without a `with` block joins the whole side stream."""
        cur = torch.cuda.current_stream(self.rt.device)
        if self._done is not None:
            cur.wait_event(self._done)
        else:
            cur.wait_stream(self.rt.side_stream)


_default: Optional[Runtime] = None


def get_runtime() -> Runtime:
    global _default
    if _default is None:
        _default = Runtime()
    return _default


def set_runtime(rt: Optional[Runtime]) -> None:
    global _default
    _default = rt


def dt_of(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return SG_F32
    if t.dtype == torch.bfloat16:
        return SG_BF16
    raise TypeError("unsupported tensor dtype {}".format(t.dtype))
