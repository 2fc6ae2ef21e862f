"""The image loop of the reference's test.py / validate() (super-resolve one image, score it with NIQE, next image) against
the list form (Generator.infer_many + iqa.niqe_many) on seeded lists of differently sized LR images. For each list size it
reports, with CUDA events after every shape has run once:
  1. the per-image NIQE loop over the SR images against one niqe_many call;
  2. the whole loop per image (infer + NIQE);
  3. the same work as infer_many + niqe_many;
  4. the share of NIQE in 2 and in 3.
The generator has seeded random weights (the scores are not meaningful image quality, the work is the same) and the
pristine statistics are synthetic. Also reports the largest relative difference between the scores of the two paths.
Prints one JSON line per list size with the card's name and power limit read in the same run.

    python tools/time_test_loop.py [--counts 14,64] [--lo 64] [--hi 160] [--crop-border 4] [--reps 5]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import resr_b200
from oracle import generator as og
from tools.time_infer_many import card, timed


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--counts", default="14,64", help="list sizes, comma separated")
    ap.add_argument("--lo", type=int, default=64, help="smallest LR side")
    ap.add_argument("--hi", type=int, default=160, help="largest LR side")
    ap.add_argument("--crop-border", type=int, default=4)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    torch.set_grad_enabled(False)
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(og.rich_state_dict(args.seed))
    g = g.cuda().eval().assume_static_weights()
    prng = np.random.default_rng(args.seed + 1)
    a = prng.normal(0, 0.3, (36, 36))
    pristine = (prng.normal(0, 1, 36), a @ a.T + 0.05 * np.eye(36))
    metric = resr_b200.iqa.NIQE(args.crop_border, pristine)
    name = card()
    for count in [int(c) for c in args.counts.split(",")]:
        rng = np.random.default_rng(args.seed + count)
        sizes = [(int(rng.integers(args.lo, args.hi + 1)), int(rng.integers(args.lo, args.hi + 1))) for _ in range(count)]
        gen = torch.Generator(device="cuda").manual_seed(args.seed + count)
        xs = [torch.rand(1, 3, h, w, device="cuda", generator=gen) for h, w in sizes]
        srs = g.infer_many(xs)

        def niqe_loop():
            return torch.stack([metric(sr) for sr in srs]).cpu()

        def niqe_list():
            return metric.forward_many(srs).cpu()

        def test_loop():                                      # test.py: per image, SR then NIQE
            return torch.stack([metric(g.infer(x)) for x in xs]).cpu()

        def test_list():
            return metric.forward_many(g.infer_many(xs)).cpu()

        fns = {"niqe_loop": niqe_loop, "niqe_list": niqe_list, "test_loop": test_loop, "test_list": test_list}
        warm = {k: fn() for k, fn in fns.items()}             # every shape once: plans, modules, solver set-up
        t = {k: [] for k in fns}
        for _ in range(args.reps):                            # alternate the paths so that clock drift hits all of them
            for k, fn in fns.items():
                t[k] += timed(fn, 1)
        best = {k: min(v) for k, v in t.items()}
        rel = ((warm["niqe_list"] - warm["niqe_loop"]).abs() / warm["niqe_loop"].abs()).max().item()
        rel_test = ((warm["test_list"] - warm["test_loop"]).abs() / warm["test_loop"].abs()).max().item()
        print(json.dumps({
            "card": name, "images": count, "lr_sides": [args.lo, args.hi], "crop_border": args.crop_border, "seed": args.seed,
            "sr_mpix": sum(16 * h * w for h, w in sizes) / 1e6, "ms": t,
            "niqe_loop_per_image_ms": best["niqe_loop"] / count, "niqe_list_per_image_ms": best["niqe_list"] / count,
            "niqe_speedup": best["niqe_loop"] / best["niqe_list"],
            "test_loop_per_image_ms": best["test_loop"] / count, "test_list_per_image_ms": best["test_list"] / count,
            "test_speedup": best["test_loop"] / best["test_list"],
            "niqe_share_of_loop": best["niqe_loop"] / best["test_loop"], "niqe_share_of_list": best["niqe_list"] / best["test_list"],
            "max_rel_score_diff_list_vs_loop": rel, "max_rel_score_diff_test_list_vs_loop": rel_test}))


if __name__ == "__main__":
    main()
