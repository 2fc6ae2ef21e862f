"""One process, several GPUs: model.MultiDeviceInference on 1, 2, 4 and 8 devices (as many as are visible).
  cfg5: one 2048^2 LR image -> 8192^2, as an fp32 tensor (infer_large) and as a u8 image (infer_u8_large), from and to
        pinned host memory, with the default band plan (at least two bands per replica);
  list: the seeded 64-image list of tools/time_test_loop.py (LR sides 64..160) as u8 images from pinned host memory
        (infer_u8_many), at the default canvas budget and at an eighth of it (more canvases to deal).
Host clock around the whole call, which returns once every replica's streams are synchronised. Every configuration runs
once first (every band and canvas shape: plans, workspaces, modules), then five repetitions alternate the configurations.
Prints every card's name and power limit read in the same run and, per configuration, the host time a replica's worker
spends per band or canvas before its final synchronise (this includes waiting on a full launch queue when the GPU is
the bottleneck), and separately the host time to enqueue one middle band's forward on an idle GPU. Checks that the cfg5
fp32 result equals infer_tiled with the same band plan on one GPU and that the list results do not depend on the device
count.

    python tools/time_multi_device.py [--counts 1,2,4,8] [--size 2048] [--reps 5]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import resr_b200
from oracle import generator as og


def cards():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out.splitlines() if out else [torch.cuda.get_device_name(i) for i in range(torch.cuda.device_count())]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--counts", default="1,2,4,8", help="device counts, comma separated (those above the visible count are skipped)")
    ap.add_argument("--size", type=int, default=2048, help="LR side of the cfg5 image")
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs CUDA devices")
    torch.set_grad_enabled(False)
    M = resr_b200.model
    visible = torch.cuda.device_count()
    counts = [n for n in (int(c) for c in args.counts.split(",")) if n <= visible]
    gen = M.Generator(3, 3, 4)
    gen.load_state_dict(og.rich_state_dict(args.seed))
    gen = gen.cuda().eval().assume_static_weights()
    mds = {n: M.MultiDeviceInference(gen, list(range(n))) for n in counts}

    s = args.size
    g = torch.Generator().manual_seed(args.seed + 7)
    img = torch.randint(0, 256, (s, s, 3), generator=g, dtype=torch.uint8).pin_memory()
    x = (img.permute(2, 0, 1).float() / 255.0).unsqueeze(0).contiguous().pin_memory()
    out = torch.empty((1, 3, 4 * s, 4 * s)).pin_memory()
    out8 = torch.empty((4 * s, 4 * s, 3), dtype=torch.uint8).pin_memory()
    rng = np.random.default_rng(args.seed + args.images)       # tools/time_test_loop.py's list of this size
    sizes = [(int(rng.integers(64, 161)), int(rng.integers(64, 161))) for _ in range(args.images)]
    imgs = [torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8).pin_memory() for h, w in sizes]
    budgets = (M.CANVAS_MAX_PIXELS, M.CANVAS_MAX_PIXELS // 8)

    work = {}
    for n in counts:
        md = mds[n]
        work[(n, "cfg5_fp32")] = lambda md=md: md.infer_large(x, out=out)
        work[(n, "cfg5_u8")] = lambda md=md: md.infer_u8_large(img, out=out8)
        for b in budgets:
            work[(n, f"list_u8_budget{b}")] = lambda md=md, b=b: md.infer_u8_many(imgs, max_pixels=b)
    lists = {}
    for key, fn in work.items():                                # every shape once
        r = fn()
        if key[1].startswith("list"):
            lists[key] = r
    ms = {key: [] for key in work}
    enq = {key: [] for key in work}
    for _ in range(args.reps):                                  # alternate so that clock drift hits every configuration
        for key, fn in work.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            ms[key].append((time.perf_counter() - t0) * 1e3)
            per = [sec * 1e3 / items for _, items, sec in mds[key[0]].last_enqueue if items]
            enq[key].append(max(per))

    idle = {}
    for name, u8 in (("cfg5_fp32", False), ("cfg5_u8", True)):
        for n in counts:
            rows = M.default_band_rows(s, s, n) + 32          # a middle band's window: interior + two 16-row halos
            rep, dev = mds[n]._replicas[0], mds[n].devices[0]
            win = torch.zeros((1, rows, s, 3), dtype=torch.uint8, device=dev) if u8 else torch.zeros((1, 3, rows, s), device=dev)
            fn = rep.infer_u8 if u8 else rep.infer
            fn(win)                                             # the plan of this shape
            t = []
            for _ in range(args.reps):
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                fn(win)
                t.append((time.perf_counter() - t0) * 1e3)
            torch.cuda.synchronize(dev)
            idle[(n, name)] = min(t)
    same_list = {b: all(all(torch.equal(a, c) for a, c in zip(lists[(n, f"list_u8_budget{b}")], lists[(counts[0], f"list_u8_budget{b}")]))
                        for n in counts) for b in budgets}
    equal_tiled = {}
    for n in counts:
        y = mds[n].infer_large(x, out=out)
        rows = M.default_band_rows(s, s, n)
        ref = M.infer_tiled(gen, x.cuda(), rows, s, 16)[0]
        equal_tiled[n] = bool(torch.equal(y, ref.cpu()))
        del ref
        torch.cuda.empty_cache()

    print(json.dumps({"cards": cards(), "visible": visible, "cfg5_lr": [s, s], "list_images": args.images,
                      "list_lr_mpix": sum(h * w for h, w in sizes) / 1e6,
                      "list_canvases": {b: len(M.canvas_groups(sizes, b)) for b in budgets}}))
    for (n, name), t in ms.items():
        bands = len(M.plan_tiles(s, s, M.default_band_rows(s, s, n), s, 16)) if name.startswith("cfg5") else None
        row = {"devices": n, "workload": name, "ms": [round(v, 2) for v in t], "best_ms": round(min(t), 2),
               "median_ms": round(float(np.median(t)), 2), "host_ms_per_item_in_call_worst_replica": round(min(enq[(n, name)]), 3)}
        if bands is not None:
            row.update(bands=bands, band_rows=M.default_band_rows(s, s, n), lr_mpix_per_s=round(s * s / (min(t) * 1e3), 1),
                       scaling_vs_1=round(min(ms[(counts[0], name)]) / min(t), 2),
                       enqueue_one_band_idle_gpu_ms=round(idle[(n, name)], 3))
            if name == "cfg5_fp32":
                row["equals_infer_tiled"] = equal_tiled[n]
        else:
            row["equals_fewest_devices"] = same_list[int(name.rsplit("budget", 1)[1])]
        print(json.dumps(row))


if __name__ == "__main__":
    main()
