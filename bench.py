#!/usr/bin/env python
"""Benchmark of the ScrabbleGAN train step (BASELINE.json metric: train images/sec on 32 x 16*len word batches).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dtype bf16|tf32|fp32] [--length L] [--batch B] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...     (N > 1)
    python bench.py --impl reference ...      # the reference's own CPU path (torch-CPU restatement, see below)

Workload (BASELINE.json configs[3], SURVEY.md section 8d C4): one full G + D + R train step with gradient balancing
(hinge loss, Adam x3, z from noise), batch 64 PER GPU, fixed 5-character synthetic words for both the real and the
fake batch (32x80 images, i.e. also the shape of configs[0], so both arms run the same config), data-parallel
(weak scaling) with NCCL gradient sum-all-reduce and cross-replica BN statistics.  Synthetic data, random-init
weights (there is no network for datasets / checkpoints).

One JSON line is printed by rank 0:
  value        images/s, whole job, inputs already resident in HBM, K steps timed with CUDA events, max over ranks
  e2e          the same metric through the public train_step API with HOST (pinned numpy) inputs: H2D copies of
               images / labels / noise and the D2H read of the 16 statistics are inside the timed region
  roofline     the dominant kernel (tcgen05 implicit-GEMM conv) on its largest launch shape, timed live with CUDA
               events inside the timed region; `step` adds the whole-step algorithmic TFLOP/s
  cpu_baseline the reference's CPU path on this box's host cores (bounded sample), rank 0 only

--dump-outputs DIR writes what the last timed step computed as DIR/*.npy (see dump_outputs); the inputs and initial
weights are seeded, so two builds run with the same arguments can be compared file by file.

The reference arm (--impl reference): TensorFlow / Keras / gin are not installable in this image (no network, not
in the wheelhouse), so `baseline/_ref` cannot be produced; following the tier contract the arm times the torch-CPU
restatement of the reference step (oracle/sgan_oracle.py, "port") with all host threads on a bounded sample."""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# forward GFLOP per image (BASELINE.md section 3 / SURVEY.md section 8d), linear in L except attention
GF_GC = {1: 0.326, 5: 1.736, 10: 3.734}
GF_D = {1: 1.986, 5: 9.938, 10: 19.891}
GF_R = {1: 0.196, 5: 0.988, 10: 1.977}


def _interp(tab, l):
    if l in tab:
        return tab[l]
    ks = sorted(tab)
    lo = max(k for k in ks if k <= l) if l >= ks[0] else ks[0]
    hi = min(k for k in ks if k >= l) if l <= ks[-1] else ks[-1]
    if lo == hi:
        return tab[lo] * l / lo
    return tab[lo] + (tab[hi] - tab[lo]) * (l - lo) / (hi - lo)


def step_gflop_per_image(lr, lf, executed=True):
    """Mode A (G+D+R) FLOPs of one step per image: fwd + 2x fwd for a trainable backward + 1x for a frozen one.
    executed=False: the reference's own tapes (data_utils.py:449-468: D is back-propagated twice over the fake images, once
    for its filter gradients and once, frozen, for the G loss).  executed=True (what every TFLOP/s figure of this file uses):
    libsgan back-propagates D once for both losses (Discriminator.backward_merged), so the frozen D pass is not executed."""
    gc, dlf, dlr, rlf, rlr = _interp(GF_GC, lf), _interp(GF_D, lf), _interp(GF_D, lr), _interp(GF_R, lf), _interp(GF_R, lr)
    total = (gc + dlf + rlf + dlr + rlr) + 2 * (dlr + dlf) + 2 * rlr + (dlf + rlf) + 2 * gc
    return total - dlf if executed else total


def workload_name(batch, length):
    return ("ScrabbleGAN G+D+R train step, hinge + gradient balancing, Adam x3, fixed %d-char words (32x%d), batch %d per GPU"
            % (length, 16 * length, batch))


def load_traffic():
    """DRAM bytes (read + write) of the dominant kernel's largest launch, from the committed `ncu --set full` capture."""
    p = os.path.join(ROOT, "profiles", "top_kernel_traffic.json")
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "bf16_tflops": d.get("bf16_tflops", 1590.0),
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the torch-CPU restatement of the reference step
# ----------------------------------------------------------------------------------------------------
def cpu_reference_step_time(batch, length, steps, warmup, threads=None, budget_s=None):
    """Times the torch-CPU restatement of the reference step (oracle/sgan_oracle.py) on `threads` host threads.  With
    `budget_s`, the sample batch is halved (from `batch`) until warmup + steps fit the budget, judged from one probe step at
    batch 8.  Returns (seconds per step, threads, batch actually used)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import sgan_oracle as O
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    dt = torch.float32
    P0 = {"G": O.make_generator_params(1, dt), "D": O.make_discriminator_params(2, dt), "R": O.make_recognizer_params(3, dt)}

    def data(b):
        g = torch.Generator().manual_seed(1234)
        return (torch.rand(b, 32, 16 * length, 1, generator=g) * 2 - 1, torch.randint(0, 52, (b, length), generator=g),
                torch.randint(0, 52, (b, length), generator=g), torch.randn(b, 128, generator=g))

    if budget_s is not None and batch > 8:
        images, labels, fake, z = data(8)
        O.train_step(P0, {}, images, labels, fake, z, loss_fn="hinge", apply_gradient_balance=True)       # page in / warm the allocator
        t0 = time.perf_counter()
        O.train_step(P0, {}, images, labels, fake, z, loss_fn="hinge", apply_gradient_balance=True)
        per_img = (time.perf_counter() - t0) / 8
        while batch > 8 and per_img * batch * (steps + warmup) > budget_s:
            batch //= 2
    images, labels, fake, z = data(batch)
    P, opt, times = P0, {}, []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        _, P, opt = O.train_step(P, opt, images, labels, fake, z, loss_fn="hinge", apply_gradient_balance=True)
        t1 = time.perf_counter()
        if i >= warmup:
            times.append(t1 - t0)
    return sum(times) / len(times), threads, batch


def run_reference_arm(args):
    """The reference's own CPU path, timed on the box's host cores: rank 0 only.  The step runs at the arm's full per-GPU
    batch when warmup + steps fit ~4 minutes (they do at the driver's 20 + 5 steps on 16 cores), else on the largest
    power-of-two fraction of it that does; `same_config` / `cpu_baseline.sample` say which."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    warm = max(min(args.warmup, 2), 1)
    want_b = args.ref_batch if args.ref_batch > 0 else args.batch
    t, threads, sample_b = cpu_reference_step_time(want_b, args.length, args.steps, warm, budget_s=args.ref_budget_s)
    value = sample_b / t
    same = sample_b == args.batch
    line = {"impl": "reference", "metric": "train images/sec (32x16*len words)", "value": value, "unit": "images/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": warm, "ms_per_step": t * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(sample_b, args.length) + ("" if same else " [bounded CPU sample of the batch-%d workload]" % args.batch),
                       "batch_per_gpu": sample_b, "global_batch": sample_b, "word_len": args.length,
                       "parallelism": "host cores (rank 0 only; one CPU process whatever --gpus says)"},
            "same_config": same,
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port",
                             "sample": "batch %d per step of the 32x%d workload (torch-CPU fp32 restatement of the reference "
                                       "step, oracle/sgan_oracle.py; TensorFlow is not installable here)" % (sample_b, 16 * args.length)},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# secondary workloads (BASELINE.json configs[1] and configs[2]); single GPU, eager, CUDA events
# ----------------------------------------------------------------------------------------------------
def run_secondary(args):
    import numpy as np
    import torch
    runtime = importlib.import_module("scrabble-gan_b200.runtime")
    na = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture")
    rt = runtime.Runtime(device=int(os.environ.get("LOCAL_RANK", "0")), mode=args.dtype)
    runtime.set_runtime(rt)
    rng = np.random.RandomState(1234)
    in_dim = (32, 160, 1)
    if args.workload == "inference":
        G = na.make_generator(128, in_dim, (32, 8192), None, "B3", 52, vis_model=False, rt=rt)
        lengths = rng.randint(1, 11, size=256)
        buckets = [(l, int((lengths == l).sum())) for l in range(1, 11) if (lengths == l).any()]
        data = [(torch.from_numpy(rng.standard_normal(size=(n, 128)).astype(np.float32)).to(rt.device),
                 torch.from_numpy(rng.randint(0, 52, size=(n, l)).astype(np.int32)).to(rt.device)) for l, n in buckets]

        def one():
            return [G([z, y], training=False) for z, y in data]
        images, name = 256, "generator-only inference (run_inference path, training=False), 256 words of 1-10 chars in %d length buckets" % len(buckets)
    else:
        R = na.make_recognizer(in_dim, None, 81, vis_model=False, rt=rt)
        x = torch.from_numpy(rng.uniform(-1, 1, size=(256, 32, 160, 1)).astype(np.float32)).to(rt.device)
        y = torch.from_numpy(rng.randint(0, 80, size=(256, 10)).astype(np.int32)).to(rt.device)

        def one():
            R.store.zero_grad()
            loss, cache = R.forward(rt, x, y)
            R.backward(rt, cache, None, wgrad=True, want_dx=False)
            return loss
        images, name = 256, "recognizer CRNN + CTC loss fwd/bwd, batch 256, 32x160 images, 81 classes"
    for _ in range(max(args.warmup, 3)):
        one()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = rt.launch_count()
    e0.record()
    for _ in range(args.steps):
        one()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    print(json.dumps({"metric": "images/sec", "value": images / (ms * 1e-3), "unit": "images/s", "n_gpus": 1, "steps": args.steps,
                      "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "dtype": args.dtype, "data": "synthetic",
                      "config": {"workload": name}, "gpu_launches": int(rt.launch_count() - n0)}), flush=True)



# ----------------------------------------------------------------------------------------------------
# secondary legs of the one driver-visible line (SURVEY.md section 8d: C4 at L = 10 and with per-step random lengths, the
# fp32-class tf32 mode, C2 generator inference, C3 recogniser + CTC, C5 at 128 per GPU) and the data-parallel check
# ----------------------------------------------------------------------------------------------------
def _timed(torch, fn, steps, barrier):
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    barrier()
    return e0.elapsed_time(e1) / steps


def secondary_legs(args, rt, mods, nets, opts, barrier, world, rank):
    import numpy as np
    import torch
    du, dp, na = mods["du"], mods["dp"], mods["na"]
    G, D, R, gan = nets
    g_opt, d_opt, r_opt, w_opt, loss_fn, disc_iters, agb = opts
    B = args.batch
    rng = np.random.RandomState(4321 + rank)
    out = {}

    def data(b, lr, lf):
        return tuple(t.to(rt.device) for t in (
            torch.from_numpy(rng.uniform(-1, 1, size=(b, 32, 16 * lr, 1)).astype(np.float32)),
            torch.from_numpy(rng.randint(0, 52, size=(b, lr)).astype(np.int32)),
            torch.from_numpy(rng.randint(0, 52, size=(b, lf)).astype(np.int32)),
            torch.from_numpy(rng.standard_normal(size=(b, 128)).astype(np.float32))))

    def step_on(bufs, i, b):
        imgs, labels, fake, z = bufs
        return du.train_step(0, i, 1, imgs, labels, D, R, None, gan, g_opt, d_opt, r_opt, w_opt, None, b, 128, loss_fn, disc_iters, agb,
                             None, 10, "", fake_labels=fake, noise=z, return_device_stats=True)

    def leg_fixed(name, b, length, steps, note):
        bufs = data(b, length, length)
        for i in range(4):
            step_on(bufs, i, b)
        ms = _timed(torch, lambda i: step_on(bufs, i, b), steps, barrier)
        gf = step_gflop_per_image(length, length)
        out[name] = {"workload": note, "ms_per_step": ms, "images_per_s": b * world / (ms * 1e-3), "steps": steps, "dtype": rt.mode,
                     "algorithmic_tflops_per_gpu": gf * 1e-3 * b / (ms * 1e-3)}

    if world == 1:
        leg_fixed("c4_fixed_L10", B, 10, 10, "full G+D+R step, batch %d, fixed 10-char words (32x160)" % B)
        # per-step (L_real, L_fake) ~ U{1..10} from the shared-seed schedule every rank agrees on (SURVEY 8d C4).  Every
        # signature gets its own CUDA graph out of one shared memory pool; the warm-up below visits each pair of the timed
        # schedule until it is captured (one eager call + the capturing call), as the first epoch of a training run does.
        steps = 60
        sched = [dp.length_schedule(s, seed=1234) for s in range(steps)]
        pairs = sorted(set(sched))
        bufs = {pr: data(B, pr[0], pr[1]) for pr in pairs}
        old_warm = du.GRAPH_WARMUP
        du.GRAPH_WARMUP = 1
        t0 = time.perf_counter()
        for pr in pairs:
            for i in range(3):
                step_on(bufs[pr], i, B)
        torch.cuda.synchronize()
        warm_s = time.perf_counter() - t0
        r0 = rt.replayed_launches
        n0 = rt.launch_count()
        ms = _timed(torch, lambda i: step_on(bufs[sched[i]], i, B), steps, barrier)
        replayed = rt.replayed_launches - r0
        total = rt.launch_count() - n0
        du.GRAPH_WARMUP = old_warm
        gf = sum(step_gflop_per_image(a, b_) for a, b_ in sched) / steps
        out["c4_random_L"] = {"workload": "full G+D+R step, batch %d, per-step (L_real, L_fake) ~ U{1..10} (dp.length_schedule, seed 1234)" % B,
                              "ms_per_step": ms, "images_per_s": B / (ms * 1e-3), "steps": steps, "dtype": rt.mode,
                              "distinct_length_pairs": len(pairs), "fused_pairs": sum(1 for a, b_ in pairs if a == b_),
                              "launches_replayed_from_graphs_frac": replayed / max(total, 1), "warmup_s_all_pairs": warm_s,
                              "mean_gflop_per_image": gf, "algorithmic_tflops_per_gpu": gf * 1e-3 * B / (ms * 1e-3)}
        # fp32-class mode: fp32 storage, tf32 tensor-core operands for forward, dgrad AND wgrad
        mode0 = rt.mode
        rt.set_mode("tf32")
        try:
            leg_fixed("c4_tf32_L5", B, args.length, 10, "full G+D+R step, batch %d, fixed %d-char words, tf32 operands / fp32 storage" % (B, args.length))
        finally:
            rt.set_mode(mode0)
        # C2: generator-only inference, 256 words of 1-10 characters in length buckets (run_inference path, training=False)
        lengths = rng.randint(1, 11, size=256)
        buckets = [(l, int((lengths == l).sum())) for l in range(1, 11) if (lengths == l).any()]
        inf = [(torch.from_numpy(rng.standard_normal(size=(n, 128)).astype(np.float32)).to(rt.device),
                torch.from_numpy(rng.randint(0, 52, size=(n, l)).astype(np.int32)).to(rt.device)) for l, n in buckets]
        for _ in range(3):
            [G([z, y], training=False) for z, y in inf]
        ms = _timed(torch, lambda i: [G([z, y], training=False) for z, y in inf], 10, barrier)
        out["c2_inference"] = {"workload": "generator-only inference (training=False), 256 words of 1-10 chars in %d length buckets" % len(buckets),
                               "ms_per_batch": ms, "images_per_s": 256 / (ms * 1e-3), "dtype": rt.mode}
        # C3: recogniser CRNN + CTC forward + backward, batch 256, 32x160, 80-class alphabet (81 outputs)
        R81 = na.make_recognizer((32, 160, 1), None, 81, vis_model=False, rt=rt, seed=9)
        x = torch.from_numpy(rng.uniform(-1, 1, size=(256, 32, 160, 1)).astype(np.float32)).to(rt.device)
        y = torch.from_numpy(rng.randint(0, 80, size=(256, 10)).astype(np.int32)).to(rt.device)

        def r_step(i):
            R81.store.zero_grad()
            loss, cache = R81.forward(rt, x, y)
            R81.backward(rt, cache, None, wgrad=True, want_dx=False)
        for i in range(3):
            r_step(i)
        ms = _timed(torch, r_step, 10, barrier)
        out["c3_recognizer_ctc"] = {"workload": "recognizer CRNN + CTC fwd/bwd, batch 256, 32x160 images, 81 outputs", "ms_per_batch": ms,
                                    "images_per_s": 256 / (ms * 1e-3), "dtype": rt.mode,
                                    "algorithmic_tflops": 3 * 1.978 * 1e-3 * 256 / (ms * 1e-3)}
    else:
        # C5: bf16, 128 per GPU (global 1024 at 8 GPUs), sync-BN + gradient all-reduce
        leg_fixed("c5_b128_per_gpu", 128, args.length, 10,
                  "bf16 full step, 128 per GPU x %d GPUs = global batch %d, sync-BN + NCCL gradient all-reduce" % (world, 128 * world))
    return out


def dp_check(args, rt, mods, nets, world, rank):
    """Driver-visible data-parallel correctness (tests/test_dp_gpu.py cannot run on the 1-GPU test box):
    (i) after the timed steps every replica holds bit-identical weights; (ii) one fp32 step on tiny shapes: N replicas on
    their shards == ONE replica on the concatenated batch (gradients, relative L2 per network)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    du, na, nl, optim, runtime = mods["du"], mods["na"], mods["nl"], mods["optim"], mods["runtime"]
    res = {}
    sums = []
    for m in nets[:3]:
        w = m.store.w
        sums += [int(w.view(torch.int32).to(torch.int64).sum().item()), int(m.store.s.view(torch.int32).to(torch.int64).sum().item())]
    t = torch.tensor(sums, device=rt.device, dtype=torch.int64)
    allt = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(allt, t)
    res["weights_bit_identical_across_replicas"] = bool(all(torch.equal(allt[0], a) for a in allt))

    graph0, mode0 = du.GRAPH_ENABLED, rt.mode
    du.GRAPH_ENABLED = False
    rt.set_mode("fp32")
    try:
        b, l, in_dim = 2, 2, (32, 160, 1)

        def shard(r):
            g = np.random.RandomState(777 + r)
            return (g.uniform(-1, 1, size=(b, 32, 16 * l, 1)).astype(np.float32), g.randint(0, 52, size=(b, l)).astype(np.int32),
                    g.randint(0, 52, size=(b, l)).astype(np.int32), g.standard_normal(size=(b, 128)).astype(np.float32))

        def run(rt_, data, bsz):
            G = na.make_generator(128, in_dim, (32, 8192), None, "B3", 52, vis_model=False, rt=rt_, seed=12)
            D = na.make_discriminator(in_dim, None, "B1", vis_model=False, rt=rt_, seed=11)
            R = na.make_recognizer(in_dim, None, 53, vis_model=False, rt=rt_, seed=13)
            for m in (G, D):
                for v in m.store.vars:
                    if v.name.endswith(".sigma"):
                        v.assign(np.array([0.1], np.float32))
            gan = na.make_gan(G, D, R, None, vis_model=False)
            g_opt, d_opt, r_opt, w_opt, loss_fn, disc_iters, agb = optim.setup_optimizer(2e-4, 2e-4, 2e-4, 2e-4, 0.0, 0.999, nl.hinge, 1, 1, 0)
            imgs, labels, fake, z = data
            stats = du.train_step(0, 0, 1, imgs, labels, D, R, None, gan, g_opt, d_opt, r_opt, w_opt, None, bsz, 128, loss_fn, disc_iters,
                                  agb, None, 10, "", fake_labels=fake, noise=z)
            return stats, [m.store.g.clone() for m in (G, D, R)]

        stats_dp, g_dp = run(rt, shard(rank), b)
        rt1 = runtime.Runtime(device=rt.device_index, mode="fp32")          # a single-replica runtime on the same GPU
        parts = [shard(r) for r in range(world)]
        big = tuple(np.concatenate([p[i] for p in parts], axis=0) for i in range(4))
        stats_1, g_1 = run(rt1, big, b * world)
        errs = {}
        for name, a, e in zip("GDR", g_dp, g_1):
            errs[name] = float(((a.double() - e.double()).norm() / e.double().norm().clamp_min(1e-30)).item())
        worst = torch.tensor([max(errs.values()), max(abs(x - y) / max(abs(y), 1e-2) for x, y in zip(stats_dp, stats_1))], device=rt.device,
                             dtype=torch.float64)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        res["bigbatch_step_fp32"] = {"shapes": "batch %d per replica, %d-char words" % (b, l), "grad_rel_l2_rank0": errs,
                                     "grad_rel_l2_max_over_ranks": float(worst[0]), "stats_rel_max_over_ranks": float(worst[1]),
                                     "ok": bool(worst[0] <= 1e-3 and worst[1] <= 1e-3)}
    finally:
        du.GRAPH_ENABLED = graph0
        rt.set_mode(mode0)
        runtime.set_runtime(rt)
    return res


DUMP_WEIGHT_SAMPLE = 1 << 20      # weights per network in --dump-outputs (G, D and R hold 16 M, 37 M and 5.6 M)


def dump_outputs(out_dir, stats, nets):
    """Writes what the last timed step computed: `train_step_stats.npy`, the 16 statistics train_step returns (in
    data_utils.STAT_NAMES order), and for each of G, D, R the state the step leaves behind: `<net>_weights.npy`, a fixed
    seeded sample of the trainable weights (the same indices on every run), and `<net>_bn_moving_stats.npy`, every BN
    moving mean and variance.  All float32, about 12 MiB in all."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "train_step_stats.npy"), stats.detach().float().cpu().numpy())
    for name, m in zip("GDR", nets):
        w = torch.cat([v.data.reshape(-1) for v in m.store.vars if v.trainable])
        idx = np.sort(np.random.default_rng(0).choice(w.numel(), min(DUMP_WEIGHT_SAMPLE, w.numel()), replace=False))
        np.save(os.path.join(out_dir, name + "_weights.npy"), w[torch.from_numpy(idx).to(w.device)].cpu().numpy())
        moving = [v.data.reshape(-1) for v in m.store.vars if not v.trainable]
        if moving:
            np.save(os.path.join(out_dir, name + "_bn_moving_stats.npy"), torch.cat(moving).cpu().numpy())

# ----------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default=os.environ.get("SGAN_MODE", "bf16"), choices=["bf16", "tf32", "fp32"])
    ap.add_argument("--batch", type=int, default=64, help="per-GPU batch")
    ap.add_argument("--length", type=int, default=5, help="word length (real and fake)")
    ap.add_argument("--ref-batch", type=int, default=0, help="CPU batch of the reference arm (0 = the arm's own --batch)")
    ap.add_argument("--ref-budget-s", type=float, default=240.0, help="the reference arm halves its batch until warmup+steps fit this")
    ap.add_argument("--cpu-baseline-batch", type=int, default=16, help="bounded sample batch of the in-line cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="keep train_step eager (no CUDA-graph replay)")
    ap.add_argument("--workload", default="step", choices=["step", "inference", "recognizer"],
                    help="step = BASELINE configs[3] (default, the driver's line); inference = configs[1] (generator-only, batch "
                         "256, 1-10 char words); recognizer = configs[2] (CRNN + CTC fwd/bwd, batch 256, 32x160, 81 classes)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary legs (L=10, random lengths, tf32, C2, C3, C5) and dp_check")
    ap.add_argument("--profile-range", action="store_true",
                    help="bracket the timed steps with cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "step"):
        ap.error("--dump-outputs applies to the train-step workload of --impl b200")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.workload != "step":
        run_secondary(args)
        return

    import numpy as np
    import torch
    runtime = importlib.import_module("scrabble-gan_b200.runtime")
    na = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture")
    du = importlib.import_module("scrabble-gan_b200.bigacgan.data_utils")
    nl = importlib.import_module("scrabble-gan_b200.bigacgan.net_loss")
    optim = importlib.import_module("scrabble-gan_b200.optim")
    dp = importlib.import_module("scrabble-gan_b200.dp")

    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    rt = runtime.Runtime(device=local_rank, mode=args.dtype)
    runtime.set_runtime(rt)
    if os.environ.get("SGAN_BENCH_INDEPENDENT", "0") != "1":      # diagnostics: N replicas side by side with no exchange at all
        dp.init_data_parallel(rt)
    world, rank = rt.world_size, rt.rank
    assert world == max(args.gpus, 1) or world == 1, "launch with torchrun --nproc-per-node %d" % args.gpus

    B, L = args.batch, args.length
    in_dim = (32, 160, 1)
    G = na.make_generator(128, in_dim, (32, 8192), None, "B3", 52, vis_model=False, rt=rt)
    D = na.make_discriminator(in_dim, None, "B1", vis_model=False, rt=rt)
    R = na.make_recognizer(in_dim, None, 53, vis_model=False, rt=rt)
    gan = na.make_gan(G, D, R, None, vis_model=False)
    dp.broadcast_parameters(rt, [G, D, R])
    g_opt, d_opt, r_opt, w_opt, loss_fn, disc_iters, agb = optim.setup_optimizer(2e-4, 2e-4, 2e-4, 2e-4, 0.0, 0.999, nl.hinge, 1, 1, 0)

    rng = np.random.RandomState(1234 + rank)
    nbuf = 4       # rotate a few distinct synthetic batches
    host = []
    for _ in range(nbuf):
        imgs = torch.from_numpy(rng.uniform(-1, 1, size=(B, 32, 16 * L, 1)).astype(np.float32)).pin_memory()
        labels = torch.from_numpy(rng.randint(0, 52, size=(B, L)).astype(np.int32)).pin_memory()
        fake = torch.from_numpy(rng.randint(0, 52, size=(B, L)).astype(np.int32)).pin_memory()
        z = torch.from_numpy(rng.standard_normal(size=(B, 128)).astype(np.float32)).pin_memory()
        host.append((imgs, labels, fake, z))
    dev = [tuple(t.to(rt.device) for t in h) for h in host]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host[0])
    d2h_bytes = 16 * 4

    def step(i, bufs, device_stats):
        imgs, labels, fake, z = bufs[i % nbuf]
        return du.train_step(0, i, 1, imgs, labels, D, R, None, gan, g_opt, d_opt, r_opt, w_opt, None, B, 128, loss_fn, disc_iters,
                             agb, None, 10, "", fake_labels=fake, noise=z, return_device_stats=device_stats)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    # live timing of the dominant kernel on its largest launch shape: D.B3.conv2 (fwd and dgrad), M = B*8*2L... K = 9216
    ops = importlib.import_module("scrabble-gan_b200.ops")
    prof = {"events": [], "on": False}
    orig_conv_run = ops.conv_run

    def conv_run_timed(rt_, d, x, w_master, w_packed, bias, mask, out, w_mirror=None):
        hit = prof["on"] and (w_packed is not None or w_mirror is not None) and d.c_in == 1024 and d.c_out == 1024 and \
            d.ntaps == 9 and d.grid_h == 8
        if hit:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            orig_conv_run(rt_, d, x, w_master, w_packed, bias, mask, out, w_mirror=w_mirror)
            e1.record()
            prof["events"].append((e0, e1, 2.0 * d.n * d.grid_h * d.grid_w * d.ntaps * d.c_in * d.c_out))
        else:
            orig_conv_run(rt_, d, x, w_master, w_packed, bias, mask, out, w_mirror=w_mirror)
    ops.conv_run = conv_run_timed
    graph_default = du.GRAPH_ENABLED and not args.no_graph
    du.GRAPH_ENABLED = graph_default

    # ---- live timing of the dominant kernel: eager steps (CUDA events cannot be recorded inside a replayed graph) -------
    du.GRAPH_ENABLED = False
    for i in range(2):
        step(i, dev, True)
    prof["on"] = True
    for i in range(2):
        step(i, dev, True)
    prof["on"] = False
    barrier()
    # ... and of EVERY tensor-core conv / filter-gradient launch of two more eager steps (ops' launch tracer): the kernels'
    # averages over all their launch shapes, next to the figure of the largest shape
    rt.trace = []
    for i in range(2):
        step(i, dev, True)
    barrier()
    traced, rt.trace = rt.trace, None
    kern_all = {}
    for role, dsc, ev0, ev1 in traced:
        name = None
        if role in ("tc", "tc_direct", "tc_dual", "tc_rank1"):
            name = "k_conv_tc"
        elif role == "wgrad" and dsc["ci"] >= 32 and dsc["co"] >= 32 and args.dtype != "fp32":
            name = "k_wgrad_tc"
        if name:
            e = kern_all.setdefault(name, [0, 0.0, 0.0])
            e[0] += 1
            e[1] += ev0.elapsed_time(ev1)
            e[2] += 2.0 * dsc["m"] * dsc["k"] * dsc["co"]
    du.GRAPH_ENABLED = graph_default

    for i in range(args.warmup):
        step(i, dev, True)
    barrier()

    # ---- device-resident timing ---------------------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = rt.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if args.profile_range:
        torch.cuda.profiler.start()
    e0.record()
    for i in range(args.steps):
        last_stats = step(i, dev, True)
    e1.record()
    barrier()
    if args.profile_range:
        torch.cuda.profiler.stop()
    launches = rt.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms_dev = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:       # before any later step: a replayed graph returns the same stats buffer
        dump_outputs(args.dump_outputs, last_stats, (G, D, R))

    # ---- host-side enqueue cost of one step (queue empty before, no sync inside): tells whether the step is launch bound
    barrier()
    t0 = time.perf_counter()
    step(0, dev, True)
    host_enqueue_ms = (time.perf_counter() - t0) * 1e3
    barrier()

    # ---- end-to-end timing through the public API with host buffers ------------------------------------------------
    for i in range(2):
        step(i, host, False)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i, host, False)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0

    secondary, dpc = None, None
    if not args.no_secondary and not args.profile_range:
        mods = {"du": du, "dp": dp, "na": na, "nl": nl, "optim": optim, "runtime": runtime}
        ops.conv_run = orig_conv_run
        try:
            if world > 1:
                dpc = dp_check(args, rt, mods, (G, D, R, gan), world, rank)
            secondary = secondary_legs(args, rt, mods, (G, D, R, gan), (g_opt, d_opt, r_opt, w_opt, loss_fn, disc_iters, agb), barrier, world, rank)
        except Exception as ex:          # a secondary leg never costs the headline line
            import traceback
            secondary = {"error": repr(ex)[:300], "trace": traceback.format_exc()[-600:]}

    tt = torch.tensor([ms_dev, t_e2e * 1e3], device=rt.device, dtype=torch.float64)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = float(tt[0]), float(tt[1])

    if rank == 0:
        peaks = load_peaks()
        traffic = load_traffic()
        images = B * world * args.steps
        value = images / (ms_dev * 1e-3)
        e2e = images / (ms_e2e * 1e-3)
        gf_img = step_gflop_per_image(L, L)
        step_tflops = gf_img * 1e-3 * B / (ms_dev / args.steps * 1e-3)          # per GPU
        kern_ms = [a.elapsed_time(b) for a, b, _ in prof["events"]]
        kern_fl = [f for _, _, f in prof["events"]]
        if kern_ms:
            avg_ms = sum(kern_ms) / len(kern_ms)
            achieved = (sum(kern_fl) / len(kern_fl)) / (avg_ms * 1e-3) / 1e12
        else:
            avg_ms, achieved = None, None
        peak = peaks["bf16_tflops_sustained"]
        roofline = {"bound": "tensor", "kernel": "k_conv_tc<bf16> (tcgen05 implicit-GEMM conv), largest launch shape: D.B3.conv2 dgrad, "
                    "M=%d (the fused [fake;real] batch of the merged D backward), K=9216, N=1024; timed in 2 eager steps"
                    % (2 * B * 8 * 4 * L), "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": (achieved / peak) if achieved else None, "traffic": (traffic or {}).get("traffic_bytes"),
                    "traffic_source": (traffic or {}).get("source"), "peak_source": peaks["source"] + " (sustained bf16 cuBLAS)",
                    "launches_timed": len(kern_ms), "avg_launch_ms": avg_ms,
                    "all_launch_shapes": {k: {"launches_per_step": v[0] // 2, "avg_launch_ms": v[1] / v[0],
                                              "achieved": v[2] / (v[1] * 1e-3) / 1e12, "frac": v[2] / (v[1] * 1e-3) / 1e12 / peak}
                                          for k, v in kern_all.items()},
                    "step": {"achieved": step_tflops, "frac": step_tflops / peak, "gflop_per_image": gf_img,
                             "gflop_per_image_reference_tapes": step_gflop_per_image(L, L, executed=False),
                             "note": "executed FLOPs: one merged D backward serves the D and the G loss (the reference's tapes "
                                     "back-propagate D twice over the fake images)"}}
        line = {"metric": "train images/sec (32x16*len words)", "value": value, "unit": "images/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
                "config": {"workload": workload_name(B, L), "batch_per_gpu": B, "global_batch": B * world, "word_len": L,
                           "parallelism": "dp%d" % world, "cuda_graph": bool(graph_default and (world == 1 or du.GRAPH_DP)),
                           "l2": "no explicit flush: the per-step working set (>1 GB of activations, 0.7 GB weights+optimizer state) "
                                 "exceeds the 126 MB L2 and input batches rotate"},
                "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                        "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "host_enqueue_ms_per_step": host_enqueue_ms, "clocks": clocks, "roofline": roofline}
        if secondary is not None:
            line["secondary"] = secondary
        if dpc is not None:
            line["dp_check"] = dpc
        if world == 1 and not args.no_cpu_baseline:
            try:
                t, threads, cb = cpu_reference_step_time(args.cpu_baseline_batch, L, 2, 1)
                line["cpu_baseline"] = {"value": cb / t, "unit": "images/s", "cores": threads, "kind": "port",
                                        "sample": "2 steps at batch %d of the same 32x%d workload (torch-CPU restatement of the "
                                                  "reference train step; TensorFlow is not installable here)" % (cb, 16 * L)}
            except Exception as ex:      # the baseline is a report, never a reason to lose the GPU numbers
                line["cpu_baseline"] = {"value": None, "error": repr(ex)}
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear-down: captured CUDA graphs hold NCCL work, and destroying the process group under them can block for
        # minutes.  Everything is printed and synchronised at this point, so leave through os._exit after a last barrier.
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
