"""Throughput of Generator.infer_many (one packed-canvas forward per list) against a loop of Generator.infer over the
same seeded list of differently sized images (what test.py / validate() / inference.py do per image), with CUDA events
after every shape has run once. Also compares the outputs of the two paths at the timed sizes. Prints one JSON line with
the card's name and power limit read in the same run.

    python tools/time_infer_many.py [--count 64] [--lo 32] [--hi 160] [--reps 3] [--precision fp16]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import resr_b200
from oracle import generator as og


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(0)


def timed(fn, reps):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        torch.cuda.synchronize()
        ev0.record()
        fn()
        ev1.record()
        ev1.synchronize()
        ms.append(ev0.elapsed_time(ev1))
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--count", type=int, default=64)
    ap.add_argument("--lo", type=int, default=32, help="smallest LR side")
    ap.add_argument("--hi", type=int, default=160, help="largest LR side")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16"])
    args = ap.parse_args()
    torch.set_grad_enabled(False)
    rng = np.random.default_rng(args.seed)
    sizes = [(int(rng.integers(args.lo, args.hi + 1)), int(rng.integers(args.lo, args.hi + 1))) for _ in range(args.count)]
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(og.rich_state_dict(args.seed))
    g = g.cuda().eval().set_precision(args.precision).assume_static_weights()
    gen = torch.Generator(device="cuda").manual_seed(args.seed)
    xs = [torch.rand(1, 3, h, w, device="cuda", generator=gen) for h, w in sizes]

    many = g.infer_many(xs)                                   # warm-up: canvas plan(s)
    alone = [g.infer(x) for x in xs]                          # warm-up: one plan per shape (rebuilt as shapes alternate)
    diff = max((a - b).abs().max().item() for a, b in zip(many, alone))
    t_many = timed(lambda: g.infer_many(xs), args.reps)
    t_loop = timed(lambda: [g.infer(x) for x in xs], args.reps)
    lr_px = sum(h * w for h, w in sizes)
    pos, canvas = resr_b200._lib.canvas_pack(sizes)
    best_many, best_loop = min(t_many), min(t_loop)
    print(json.dumps({
        "card": card(), "precision": args.precision, "images": args.count, "lr_sides": [args.lo, args.hi], "seed": args.seed,
        "lr_mpix": lr_px / 1e6, "canvas": canvas, "canvas_fill": lr_px / (canvas[0] * canvas[1]),
        "infer_many_ms": t_many, "infer_loop_ms": t_loop,
        "infer_many_images_per_s": args.count / best_many * 1e3, "infer_loop_images_per_s": args.count / best_loop * 1e3,
        "infer_many_lr_mpix_per_s": lr_px / best_many / 1e3, "infer_loop_lr_mpix_per_s": lr_px / best_loop / 1e3,
        "speedup": best_loop / best_many, "max_abs_many_vs_loop": diff}))


if __name__ == "__main__":
    main()
