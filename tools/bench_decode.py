"""Timing of reading words back with the recogniser (scrabble-gan_b200/decode.py), with CUDA events after warm-up:
  (a) softmax + greedy CTC decoding + edit distance alone, at config 3's shape (B = 256, T = 39, C = 81) and at B = 4096;
  (b) evaluate_recognizer on B = 256, 32x160 batches (images/s), and the three kernels' share of its device time;
  (c) evaluate_generated_words on 256 words of 1-10 characters (words/s).
Prints the card's name and power limit with the numbers.  Usage: python tools/bench_decode.py [--iters N] [--out file.json]"""
import argparse
import importlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

runtime = importlib.import_module("scrabble-gan_b200.runtime")
ops = importlib.import_module("scrabble-gan_b200.ops")
na = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture")
decode = importlib.import_module("scrabble-gan_b200.decode")

from _bench_util import card, kernel_us, timed_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rt = runtime.Runtime(device=0, mode=args.mode)
    runtime.set_runtime(rt)
    res = {"card": card(), "mode": args.mode, "iters": args.iters}
    g = torch.Generator(device=rt.device).manual_seed(0)

    # (a) the three kernels alone
    def tail(b, t=39, c=81):
        logits = torch.randn(b, t, c, device=rt.device, generator=g) * 3
        labels = torch.randint(0, c - 1, (b, 10), device=rt.device, dtype=torch.int32, generator=g)
        il = torch.full((b,), t, device=rt.device, dtype=torch.int32)
        totals = torch.zeros(4, device=rt.device, dtype=torch.int64)

        def run():
            p = ops.softmax_rows(rt, logits)
            dec, dlen, _ = ops.ctc_greedy_decode(rt, p, il)
            ops.edit_distance(rt, dec, labels, dlen, None, totals)
        return run
    for b in (256, 4096):
        res["a_tail_b%d_us" % b] = 1e3 * timed_ms(tail(b), args.iters * 4)

    # (b) evaluate_recognizer, B = 256, 32x160 (T = 39), 81 outputs
    R = na.make_recognizer((32, 160, 1), None, 81, vis_model=False, rt=rt, seed=9)
    nb = 8
    batches = [(torch.rand(256, 32, 160, 1, device=rt.device, generator=g) * 2 - 1,
                torch.randint(0, 80, (256, 10), device=rt.device, dtype=torch.int32, generator=g)) for _ in range(nb)]
    ms = timed_ms(lambda: decode.evaluate_recognizer(R, batches), max(args.iters // 5, 3), warmup=2)
    res["b_evaluate_recognizer_images_per_s"] = 256 * nb / (ms / 1e3)
    x0 = batches[0][0]
    fwd_ms = timed_ms(lambda: R._logits(rt, x0, False), args.iters)
    res["b_R_forward_ms"] = fwd_ms
    # device time of every kernel of one evaluate_recognizer pass (torch.profiler, a pass of its own): the three new kernels'
    # share, and their time against R's forward kernels (eager timing above includes the host's launch overhead)
    per = kernel_us(lambda: decode.evaluate_recognizer(R, batches), 1)
    new = ("k_softmax_rows", "k_ctc_greedy_decode", "k_edit_distance")
    t_all = sum(per.values())
    t_new = sum(t for k, t in per.items() if any(n in k for n in new))
    res["b_new_kernels_us_per_batch"] = t_new / nb
    res["b_all_kernels_us_per_batch"] = t_all / nb
    res["b_new_kernels_share_of_evaluate"] = t_new / t_all
    res["b_new_kernels_over_R_forward_kernels"] = t_new / (t_all - t_new)

    # (c) evaluate_generated_words, 256 words of 1-10 characters
    G = na.make_generator(128, (32, 160, 1), (32, 8192), None, "B3", 80, vis_model=False, rt=rt)
    gc = torch.Generator().manual_seed(1)
    lens = torch.randint(1, 11, (256,), generator=gc)
    labels = torch.randint(0, 80, (256, 10), generator=gc).int()
    for i in range(256):
        labels[i, lens[i]:] = -1
    labels = labels.to(rt.device)
    ms = timed_ms(lambda: decode.evaluate_generated_words(G, R, labels), max(args.iters // 5, 3), warmup=2)
    res["c_evaluate_generated_words_words_per_s"] = 256 / (ms / 1e3)
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
