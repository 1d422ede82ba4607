"""Timing of lexicon decoding (k_ctc_lexicon_scores, k_ctc_lexicon_topk) at config 3's shape (B = 256, T = 39, C = 81) for
lexicons of V = 1 000, 10 000 and 100 000 words of 1-10 letters, next to R's forward pass and the beam decoder at width 100
in the same run.  Each kernel's device time comes from torch.profiler (keys *_us_device); the rate is the algorithmic
state updates of the alpha recursion, B * sum_v (2 L_v + 1) * T, over the scores kernel's device time.  The launches are
preallocated calls of the C ABI.  Prints the card's name and power limit with the numbers.
Usage: python tools/bench_lexicon_decode.py [--out profiles/r05_bench_lexicon_decode.json]"""
import argparse
import importlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

_abi = importlib.import_module("scrabble-gan_b200._abi")
runtime = importlib.import_module("scrabble-gan_b200.runtime")
ops = importlib.import_module("scrabble-gan_b200.ops")
na = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture")

from _bench_util import card, device_us, r_forward_us  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rt = runtime.Runtime(device=0, mode=args.mode)
    runtime.set_runtime(rt)
    b, t, c = 256, 39, 81
    res = {"card": card(), "mode": args.mode, "calls": args.calls, "b": b, "t": t, "c": c, "sms": rt.num_sms}

    R = na.make_recognizer((32, 160, 1), None, c, vis_model=False, rt=rt, seed=9)
    g = torch.Generator(device=rt.device).manual_seed(0)
    x = torch.rand(b, 32, 160, 1, device=rt.device, generator=g) * 2 - 1
    probs = R.frame_probs(x)                                   # R's own frame probabilities as the decoders' input
    il = torch.full((b,), t, device=rt.device, dtype=torch.int32)
    ptr = _abi.ptr

    res["R_forward_us_device"] = r_forward_us(R, rt, x)

    w = 100
    dec = torch.empty((1, b, t), device=rt.device, dtype=torch.int32)
    dlen = torch.empty((1, b), device=rt.device, dtype=torch.int32)
    lp = torch.empty((b, 1), device=rt.device)
    nbytes = _abi.load().sg_ctc_beam_decode_scratch_bytes(b, t, w)
    scratch = torch.empty(nbytes, device=rt.device, dtype=torch.uint8)
    beam = lambda: _abi.call.sg_ctc_beam_decode(rt.ctx, ptr(probs), b, t, c, ptr(il), w, 1, 1, ptr(dec), ptr(dlen),  # noqa: E731
                                                ptr(lp), ptr(scratch), nbytes)
    res["beam100_us_device"] = device_us(beam, ["k_ctc_beam_decode"], args.calls)["k_ctc_beam_decode"]

    rng = np.random.default_rng(1)
    for v in (1000, 10000, 100000):
        lens_h = rng.integers(1, 11, v)
        lex_h = np.full((v, 10), -1, np.int32)
        for i, n in enumerate(lens_h):
            lex_h[i, :n] = rng.integers(0, c - 1, n)
        lex = torch.from_numpy(lex_h).to(rt.device)
        lens = ops.label_lengths(rt, lex)
        scores = torch.empty((b, v), device=rt.device)
        k = 1
        wdec = torch.empty((k, b, 10), device=rt.device, dtype=torch.int32)
        wlen = torch.empty((k, b), device=rt.device, dtype=torch.int32)
        wlp = torch.empty((b, k), device=rt.device)
        widx = torch.empty((b, k), device=rt.device, dtype=torch.int32)

        def both():
            _abi.call.sg_ctc_lexicon_scores(rt.ctx, ptr(probs), b, t, c, ptr(il), ptr(lex), ptr(lens), v, 10, ptr(scores))
            _abi.call.sg_ctc_lexicon_topk(rt.ctx, ptr(scores), b, v, ptr(lex), ptr(lens), 10, k, ptr(wdec), ptr(wlen), ptr(wlp),
                                          ptr(widx))
        d = device_us(both, ["k_ctc_lexicon_scores", "k_ctc_lexicon_topk"], args.calls)
        s_us, k_us = d["k_ctc_lexicon_scores"], d["k_ctc_lexicon_topk"]
        updates = float(b) * float(np.sum(2 * lens_h + 1)) * t
        res["v%d" % v] = {
            "scores_us_device": s_us, "topk_us_device": k_us, "state_updates": updates,
            "state_updates_per_s": updates / (s_us * 1e-6) if s_us > 0 else None,
            "pairs_per_s": b * v / (s_us * 1e-6) if s_us > 0 else None,
            "share_of_R_forward_device": (s_us + k_us) / res["R_forward_us_device"],
            "over_beam100_device": (s_us + k_us) / res["beam100_us_device"]}
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
