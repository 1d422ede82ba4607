"""Timing of the CTC beam decoder (k_ctc_beam_decode) at config 3's shape (B = 256, T = 39, C = 81) for beam_width 10 and
100, next to the greedy decoder (k_ctc_greedy_decode) and R's forward pass in the same run: CUDA events after warm-up around
back-to-back calls (keys *_host_included: host launch overhead included), and each kernel's device time from torch.profiler
(keys *_device).  The beam launches are preallocated calls of the C ABI.
Prints the card's name and power limit with the numbers.
Usage: python tools/bench_beam_decode.py [--iters N] [--out profiles/r04_bench_beam_decode.json]"""
import argparse
import importlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

_abi = importlib.import_module("scrabble-gan_b200._abi")
runtime = importlib.import_module("scrabble-gan_b200.runtime")
ops = importlib.import_module("scrabble-gan_b200.ops")
na = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture")

from _bench_util import card, device_us, r_forward_us, timed_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rt = runtime.Runtime(device=0, mode=args.mode)
    runtime.set_runtime(rt)
    b, t, c = 256, 39, 81
    res = {"card": card(), "mode": args.mode, "iters": args.iters, "b": b, "t": t, "c": c, "sms": rt.num_sms}

    R = na.make_recognizer((32, 160, 1), None, c, vis_model=False, rt=rt, seed=9)
    g = torch.Generator(device=rt.device).manual_seed(0)
    x = torch.rand(b, 32, 160, 1, device=rt.device, generator=g) * 2 - 1
    probs = R.frame_probs(x)                                   # R's own frame probabilities as the decoders' input
    il = torch.full((b,), t, device=rt.device, dtype=torch.int32)

    def beam_launch(p, lens, w):
        """One preallocated sg_ctc_beam_decode launch: no allocation in the timed loop."""
        n = p.shape[0]
        dec = torch.empty((1, n, t), device=rt.device, dtype=torch.int32)
        dlen = torch.empty((1, n), device=rt.device, dtype=torch.int32)
        lp = torch.empty((n, 1), device=rt.device)
        nbytes = _abi.load().sg_ctc_beam_decode_scratch_bytes(n, t, w)
        scratch = torch.empty(nbytes, device=rt.device, dtype=torch.uint8)
        ptr = _abi.ptr
        return lambda: _abi.call.sg_ctc_beam_decode(rt.ctx, ptr(p), n, t, c, ptr(lens), w, 1, 1, ptr(dec), ptr(dlen), ptr(lp),
                                                    ptr(scratch), nbytes)

    # CUDA events around back-to-back launches (host launch overhead included, as in r03's kernel legs), then the kernels'
    # own device time from the profiler
    res["R_forward_ms_host_included"] = timed_ms(lambda: R._logits(rt, x, False), args.iters)
    greedy = lambda: ops.ctc_greedy_decode(rt, probs, il)    # noqa: E731
    res["greedy_decode_us_host_included"] = 1e3 * timed_ms(greedy, args.iters * 4)
    res["greedy_decode_us_device"] = device_us(greedy, ["k_ctc_greedy_decode"])["k_ctc_greedy_decode"]
    res["R_forward_us_device"] = r_forward_us(R, rt, x)
    for w in (10, 100):
        fn = beam_launch(probs, il, w)
        res["beam%d_us_host_included" % w] = 1e3 * timed_ms(fn, args.iters)
        dev = device_us(fn, ["k_ctc_beam_decode"])["k_ctc_beam_decode"]
        res["beam%d_us_device" % w] = dev
        res["beam%d_share_of_R_forward_device" % w] = dev / res["R_forward_us_device"]
        res["beam%d_over_greedy_device" % w] = dev / res["greedy_decode_us_device"]
    # one CTA per sample: at B = 256 on 148 SMs the grid is under two CTAs per SM; B = 4096 keeps every SM busy, so the
    # per-sample device time at both sizes shows how much the small grid costs
    pb, ilb = probs.repeat(16, 1, 1), il.repeat(16)
    for w in (10, 100):
        res["beam%d_b256_us_per_sample_device" % w] = res["beam%d_us_device" % w] / b
        dev = device_us(beam_launch(pb, ilb, w), ["k_ctc_beam_decode"], 5)["k_ctc_beam_decode"]
        res["beam%d_b4096_us_per_sample_device" % w] = dev / (16 * b)
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
