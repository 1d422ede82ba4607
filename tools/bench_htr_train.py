"""Throughput of training the recogniser on its own (htr.train_recognizer_step) at config 3's shape: B = 256 words of L = 10
letters (32 x 160), 81 classes, bf16, Adam.  Three workloads, each timed with CUDA events over a steady-state window after a
warm-up: real words only; real words + augmentation; half generated (mixed_word_batches: 128 real + 128 words G generates in
the batch) + augmentation.  Also the augmentation kernel's device time (torch.profiler, a run of its own) and the host
enqueue time of one step (queue drained before, no synchronisation inside).  Prints the card's name and power limit with
the numbers.
Usage: python tools/bench_htr_train.py [--out profiles/r06_bench_htr_train.json]"""
import argparse
import importlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

runtime = importlib.import_module("scrabble-gan_b200.runtime")
ops = importlib.import_module("scrabble-gan_b200.ops")
optim = importlib.import_module("scrabble-gan_b200.optim")
htr = importlib.import_module("scrabble-gan_b200.htr")
na = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture")
du = importlib.import_module("scrabble-gan_b200.bigacgan.data_utils")
nl = importlib.import_module("scrabble-gan_b200.bigacgan.net_loss")

from _bench_util import card, device_us, timed_ms  # noqa: E402

AUG = dict(rotation=2.0, shear=0.3, scale=0.1, translate=2.0, p_morph=0.25)


def timed(step, warmup, steps):
    """ms per step over `steps` steps after `warmup`, from CUDA events; and the host enqueue time of one more step."""
    ms = timed_ms(step, steps, warmup)
    t0 = time.perf_counter()
    step()
    enqueue_ms = (time.perf_counter() - t0) * 1e3
    torch.cuda.synchronize()
    return ms, enqueue_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rt = runtime.Runtime(device=0, mode="bf16")
    runtime.set_runtime(rt)
    b, l, c = 256, 10, 81
    res = {"card": card(), "mode": "bf16", "b": b, "l": l, "classes": c, "warmup": args.warmup, "steps": args.steps}

    R = na.make_recognizer((32, 160, 1), None, c, vis_model=False, rt=rt, seed=9)
    opt = optim.setup_optimizer(2e-4, 2e-4, 2e-4, 2e-4, 0.0, 0.999, nl.hinge, 1, 0, 0)[2]
    g = torch.Generator(device=rt.device).manual_seed(0)
    x = torch.rand(b, 32, 16 * l, 1, device=rt.device, generator=g) * 2 - 1
    y = torch.randint(0, c - 1, (b, l), device=rt.device, generator=g, dtype=torch.int32)

    G = na.make_generator(128, (32, 160, 1), (32, 8192), None, "B3", c - 1, vis_model=False, rt=rt, seed=8)
    words = du.synthetic_random_words(l, list(range(c - 1)), words_per_bucket=256, seed=1)
    half = b // 2

    def real_batches():
        while True:
            yield x[:half], y[:half]
    mixed = htr.mixed_word_batches(real_batches(), G, words, b - half)

    workloads = {
        "real": lambda: htr.train_recognizer_step(R, opt, x, y),
        "real_augmented": lambda: htr.train_recognizer_step(R, opt, x, y, augment=AUG),
        "half_generated_augmented": lambda: htr.train_recognizer_step(R, opt, *next(mixed), augment=AUG),
    }
    for name, fn in workloads.items():
        ms, enq = timed(fn, args.warmup, args.steps)
        res[name] = {"ms_per_step_device": ms, "images_per_s": b / (ms * 1e-3), "host_enqueue_ms_per_step": enq}

    u = ops.random_(rt, rt.empty((b, 7)), normal=False)
    out = rt.empty(x.shape)
    aug = lambda: ops.word_augment(rt, x, u, None, out=out, **AUG)  # noqa: E731
    us = device_us(aug, ["k_word_augment"], 50)["k_word_augment"]
    nbytes = 2 * x.numel() * 4                              # one read and one write of every pixel, the least it can move
    res["augment_kernel"] = {"us_device": us, "pixels": x.numel(), "min_bytes": nbytes,
                             "GB_per_s_min_bytes": nbytes / (us * 1e-6) / 1e9 if us > 0 else None}
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
