#!/usr/bin/env python
"""bench.py — headline benchmark of BASELINE.json ("x4 RRDBNet LR Mpix/s + degraded pairs/s at 1/2/4/8 B200, % of roofline").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--precision fp16|bf16] [--dump-outputs DIR]

Our arm (default). One step = one RRDBNet x4 forward of the 64x3x128x128 LR batch of BASELINE.json configs[2], batch-
sharded over the N ranks (64 / N images per rank: STRONG scaling, the configuration BASELINE names; no collective on the
data path). Rank 0 prints ONE JSON line:
  value         device-timed LR Mpix/s of the whole job, inputs resident in HBM (CUDA events, max over ranks)
  e2e           the same through the host-buffer C ABI call (pinned H2D + forward + D2H inside the timed region)
  roofline      tensor-core roofline of the conv kernels against MEASURED_PEAKS.json
  cpu_baseline  (N = 1) the fp32 oracle port of the reference forward on this box's host cores (bounded sample)
  weak          (N > 1) secondary: every rank runs its own 64 images
  tiled         secondary, configs[4]: 1x3x2048x2048 -> 8192x8192 by full-width halo bands dealt to the N ranks, gathered
                into rank 0's buffer by NCCL send / recv, end to end from / to pinned host memory
  degradation   secondary, configs[1]: degraded pairs/s of the second-order pipeline (canonical plan S0, real sinc and
                mixed blur kernels), device-timed + e2e (HR from pinned host every step) + HBM and FMA rooflines + CPU port
  training      secondary, configs[3]: degradation + generator forward / L1 / backward (+ NCCL all-reduce) per GPU
`--impl reference`: the reference's own CPU implementation of the path (oracle port; /root/reference does not exist on
the GPU box) timed on the host cores, one 1x3x128x128 image per step.
`--dump-outputs DIR`: after the timed steps, the SR batch of the last timed step (rank 0's shard) goes to DIR/sr.npy in
float32 (over 48 MiB: a fixed, seeded choice of whole images, 16 of the 64 at N = 1), so that two builds can be compared
output for output: inputs and weights are seeded, identical in every run with the same arguments.
"""
import argparse
import json
import math
import os
import random
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

FLOP_PER_LR_PIXEL = 35853696.0  # SURVEY.md §8a layer table
METRIC = "x4 RRDBNet LR Mpix/s"
TOTAL_BATCH = 64                # BASELINE.json configs[2]


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    out = {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}
    if os.path.exists(p):
        d = json.load(open(p))
        out = {"hbm": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"],
               "source": "MEASURED_PEAKS.json"}
    # fp32 FMA peak measured on this pool's B200 with tools/fma_peak.cu (register-resident FFMA chains)
    f = os.path.join(ROOT, "profiles", "r02_fma_peak.json")
    out["tfma"] = json.load(open(f))["fp32_tfma_sustained"] if os.path.exists(f) else 36.2
    return out


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (NVML, 20 ms period; nvidia-smi fallback)."""

    def __init__(self, index):
        self.rows, self.stop, self.index = [], threading.Event(), index
        self.t = threading.Thread(target=self.run, daemon=True)
        self.max_mhz = None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            while not self.stop.is_set():
                mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)) if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.rows.append((mhz, r))
                self.stop.wait(0.02)
            return
        except Exception:
            pass
        q = "clocks.sm,clocks.max.sm"
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    a, b = (float(v) for v in out.split(","))
                    self.max_mhz = b
                    self.rows.append((a, 0))
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[1]
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = [n for b, n in names.items() if bits & b]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm)}


class Dist:
    """Rank plumbing: barrier + max-over-ranks of device-timed milliseconds."""

    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.device = None

    def init(self):
        import torch.distributed as dist
        torch.cuda.set_device(self.local)
        self.device = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.device)

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_ms(self, *ms):
        t = torch.tensor(list(ms), device=self.device, dtype=torch.float64)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def finish(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()


def timed(fn, steps, D, fin=None, warm=0):
    """`steps` calls of fn(k) bracketed by barrier + synchronize on both sides, CUDA events on the current stream."""
    for k in range(warm):
        fn(k)
    if fin:
        fin()
    D.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for k in range(steps):
        fn(k)
    if fin:
        fin()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    D.barrier()
    return ms


DUMP_BYTES = 48 << 20   # the arrays of one --dump-outputs run stay under 64 MB


def dump_output(out_dir, name, y):
    """Writes y (images along dim 0) as out_dir/<name>.npy in float32. An output larger than DUMP_BYTES is cut to a
    seeded choice of whole images, the same in every run; returns its shape and the images kept."""
    n, per_image = y.shape[0], y[0].numel() * 4
    idx = torch.arange(n)
    if n * per_image > DUMP_BYTES:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_BYTES // per_image].sort().values
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), y.detach()[idx.to(y.device)].float().cpu().numpy())
    return {name: {"shape": list(y.shape), "images": idx.tolist()}}


# ------------------------------------------------------------------------------------------------- CPU baselines


def cpu_generator_baseline(seconds_budget=20.0, max_iters=5):
    """Oracle port of the reference forward (plain torch fp32, all host cores) on cfg1 (1x3x128x128)."""
    from oracle import generator as og
    torch.set_num_threads(os.cpu_count() or 1)
    sd = og.random_state_dict(0)
    torch.manual_seed(0)
    x = torch.rand(1, 3, 128, 128)
    og.generator_forward(x[:, :, :32, :32], sd)  # warm-up
    times = []
    t_all = time.perf_counter()
    while len(times) < max_iters and (time.perf_counter() - t_all) < seconds_budget:
        t0 = time.perf_counter()
        og.generator_forward(x, sd)
        times.append(time.perf_counter() - t0)
    med = sorted(times)[len(times) // 2]
    return {"value": 128 * 128 / med / 1e6, "unit": "LR Mpix/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{len(times)} fp32 forwards of 1x3x128x128 (BASELINE configs[0]), median {med:.3f} s"}


def cpu_degradation_baseline(kernels_np, seconds_budget=15.0, batch=4):
    """numpy oracle port of train_realesrnet.py:267-377 (oracle/degrade.py) on `batch` HR crops of the same workload
    (canonical plan S0, the same kind of kernels), noise drawn on the fly as the reference does."""
    import resr_b200
    from oracle import degrade as od
    rng = np.random.default_rng(0)
    hr = rng.random((batch, 3, 256, 256), dtype=np.float32)
    plan = resr_b200.plan.canonical_plan_s0(batch, 256, 256, seed=0)
    plan["noise1"]["noise_color"] = None   # drawn inside the timed region, like torch.randn in the reference
    k1, k2, sk = (k[:batch] for k in kernels_np)
    od.degrade_batch(hr[:1], k1[:1], k2[:1], sk[:1], resr_b200.plan.canonical_plan_s0(1, 256, 256, seed=0), draw_rng=rng)  # warm-up (imports, FFT plans)
    times = []
    t_all = time.perf_counter()
    while len(times) < 5 and (time.perf_counter() - t_all) < seconds_budget:
        t0 = time.perf_counter()
        od.degrade_batch(hr, k1, k2, sk, plan, draw_rng=rng)
        times.append(time.perf_counter() - t0)
    med = sorted(times)[len(times) // 2]
    return {"value": batch / med, "unit": "pairs/s", "cores": 1, "kind": "port",
            "sample": f"{len(times)} runs of the numpy port on {batch}x3x256x256 HR crops (plan S0), median {med:.3f} s; "
                      "numpy / scipy.fft are single-threaded apart from BLAS inside the JPEG DCT"}


# ------------------------------------------------------------------------------------------------- degradation


def s0_kernels(B, device, seed=0):
    """kernel1 / kernel2 / sinc kernel for the canonical plan S0: mixed Gaussian-family / sinc blur kernels with the
    reference's distributions (dataset.py:81-141) synthesised on the device (resr_synthesize_kernels); the final kernel is
    a REAL sinc for every sample (S0 says "sinc"; the dataset draws one with p = 0.8)."""
    import resr_b200
    ip = resr_b200.imgproc
    P = dict(resr_b200.plan.DEGRADATION_MODEL_PARAMETERS)
    P["sinc_kernel_probability3"] = 1.0
    random.seed(seed)
    np.random.seed(seed)
    return ip.synthesize_degradation_kernels(B, P, device)


def s0_stage_bytes(B, H=256, W=256):
    """Stage-sum algorithmic bytes of S0 (SURVEY.md §8d): 4 B x (elements read + written) per EXECUTED stage. The third
    resize of S0 is a same-size resize (bit-exact identity, skipped: not counted); the Poisson stage reads its input twice
    (level census, then the noise pass) and draws its samples in the kernel (no sample tensor is read)."""
    E0 = B * 3 * H * W
    e1, e2 = E0 // 4, E0 // 16
    stages = {"usm": 2 * E0, "blur1": 2 * E0, "resize1": E0 + e1, "noise1": 2 * e1 + e1, "jpeg1": 2 * e1, "blur2": 2 * e1,
              "resize2": e1 + e2, "noise2": 2 * e2, "sinc": 2 * e2, "jpeg2": 2 * e2, "round_crop": 2 * e2}
    fma = {"usm": 4 * 51 * E0, "blur1": None, "blur2": None, "sinc": None}
    return 4 * sum(stages.values()), stages, fma


def stencil_fmas(k1, k2, sk, H=256, W=256):
    """Necessary FMAs of the S0 stencils: separable 51-tap USM (2 blurs x 2 passes) + per-sample trimmed supports."""
    def support(k):
        nz = (k != 0).nonzero()
        ext = (nz[:, 1:] - 10).abs().amax(1)
        out = torch.zeros(k.shape[0], dtype=torch.long)
        out.scatter_reduce_(0, nz[:, 0].cpu(), (2 * ext + 1).cpu(), reduce="amax")
        return out
    s1, s2, s3 = support(k1), support(k2), support(sk)
    px0, px1, px2 = 3 * H * W, 3 * H * W // 4, 3 * H * W // 16
    return float(4 * 51 * px0 * k1.shape[0] + (s1 * s1).sum() * px0 + (s2 * s2).sum() * px1 + (s3 * s3).sum() * px2)


def degradation_bench(D, steps, warmup, peaks, B=16, want_e2e=True):
    """configs[1]: B x 3 x 256 x 256 HR crops through the canonical plan S0."""
    import resr_b200
    ip = resr_b200.imgproc
    device = D.device
    H, W = 256, 256
    plan = resr_b200.plan.canonical_plan_s0(B, H, W, seed=0)
    g = torch.Generator(device="cpu").manual_seed(100 + D.rank)
    hr_host = torch.rand(B, 3, H, W, generator=g).pin_memory()
    k1, k2, sk = s0_kernels(B, device)
    pipe = ip.DegradePipeline(hr_host.to(device), k1, k2, sk, plan)
    ms = timed(lambda k: pipe(), steps, D, warm=max(3, warmup))
    out = {"ms_dev": ms}
    if want_e2e:
        # end to end: every step copies its HR batch from pinned host memory into the pipeline's input buffer and reads the
        # LR batch back; two pipelines alternate so that the copies of one step overlap the kernels of the other
        pipes = [pipe, ip.DegradePipeline(hr_host.to(device), k1, k2, sk, plan)]
        streams = [torch.cuda.Stream(device=device) for _ in range(2)]
        lr_host = [torch.empty(B, 3, H // 4, W // 4).pin_memory() for _ in range(2)]

        def step(k):
            i = k & 1
            with torch.cuda.stream(streams[i]):
                pipes[i].hr.copy_(hr_host, non_blocking=True)
                lr, _ = pipes[i]()
                lr_host[i].copy_(lr, non_blocking=True)

        def fin():
            for s in streams:
                torch.cuda.current_stream(device).wait_stream(s)

        for s in streams:
            s.wait_stream(torch.cuda.current_stream(device))
        out["ms_e2e"] = timed(step, steps, D, fin=fin, warm=4)
        out["h2d"], out["d2h"] = hr_host.numel() * 4, lr_host[0].numel() * 4
        # the same with the batch arriving as DECODED u8 images (what cv2.imread returns, dataset.py:67): 4x fewer bytes over
        # PCIe; the / 255, the augmentation (rotate / flips), BGR -> RGB and HWC -> CHW of dataset.py:67-79 run as one device
        # gather (imgproc.augment_batch) straight into the pipeline's input buffer
        img_host = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, generator=g).pin_memory()
        pipes8 = [ip.DegradePipeline(hr_host.to(device), k1, k2, sk, plan, u8_images=True) for _ in range(2)]
        random.seed(11)
        for p8 in pipes8:
            p8.augment_ops.copy_(ip.draw_augment_ops(B))

        def step_u8(k):
            i = k & 1
            with torch.cuda.stream(streams[i]):
                pipes8[i].images_u8.copy_(img_host, non_blocking=True)
                lr, _ = pipes8[i]()
                lr_host[i].copy_(lr, non_blocking=True)

        for s in streams:
            s.wait_stream(torch.cuda.current_stream(device))
        out["ms_e2e_u8"] = timed(step_u8, steps, D, fin=fin, warm=4)
        out["h2d_u8"] = img_host.numel()
    out["fma"] = stencil_fmas(k1, k2, sk)
    out["kernels_np"] = tuple(k.cpu().numpy() for k in (k1, k2, sk))
    return out


# ------------------------------------------------------------------------------------------------- training step


def training_bench(D, steps, warmup, peaks, precision="bf16", with_optimizer=True):
    """configs[3]: RealESRNet training-step core per GPU — plan-driven degradation of 16 HR crops (256^2 -> LR 64^2),
    generator forward + L1 + backward, and (world > 1) the NCCL all-reduce of the flat gradient vector. Optimizer / EMA
    are outside the north-star path (SURVEY.md §8 f1)."""
    import resr_b200
    ip = resr_b200.imgproc
    device, world = D.device, D.world
    B, H, W = 16, 256, 256
    plan = resr_b200.plan.canonical_plan_s0(B, H, W, seed=1)
    g = torch.Generator(device="cpu").manual_seed(2)
    hr = torch.rand(B, 3, H, W, generator=g).to(device)
    k1, k2, sk = s0_kernels(B, device, seed=3)   # reference-range supports (7 .. 21), real sinc
    # software-pipelined data path: the degradation of batch k + 1 (its own CUDA graph, on a data stream) runs under the
    # training step of batch k, which is latency-bound at this size and leaves SM time free; two pipelines alternate
    # (the pipelines take decoded u8 images: the end-to-end variant below uploads a fresh batch from pinned host memory per
    # step; the device-resident variant replays them on the batch that is already there)
    pipes = [ip.DegradePipeline(hr, k1, k2, sk, plan, u8_images=True) for _ in range(2)]
    img_host = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, generator=g).pin_memory()
    loss_host = torch.zeros(1).pin_memory()
    random.seed(12)
    for p_ in pipes:
        p_.images_u8.copy_(img_host)
        p_.augment_ops.copy_(ip.draw_augment_ops(B))
    torch.manual_seed(0)
    gen = resr_b200.model.Generator(3, 3, 4).to(device).train()
    gen.set_precision(precision)
    ts = resr_b200.autograd.TrainStep(gen, B, H // 4, W // 4, device, None, world)
    data = torch.cuda.Stream(device=device)
    ready = [torch.cuda.Event() for _ in range(2)]   # degradation output i is complete
    done = [torch.cuda.Event() for _ in range(2)]    # the training step that read output i has finished
    state = {"k": 0}
    cur = torch.cuda.current_stream(device)
    data.wait_stream(cur)
    with torch.cuda.stream(data):
        pipes[0]()
        ready[0].record(data)
    for e in done:
        e.record(cur)

    def step(_, e2e=False):
        k = state["k"]
        state["k"] = k + 1
        i, nxt = k & 1, (k + 1) & 1
        data.wait_event(done[nxt])
        with torch.cuda.stream(data):
            if e2e:
                pipes[nxt].images_u8.copy_(img_host, non_blocking=True)   # the next batch: decoded u8 images from pinned host memory
            pipes[nxt]()
            ready[nxt].record(data)
        cur.wait_event(ready[i])
        state["loss"], _, _ = ts.step(pipes[i].lr, pipes[i].hr_crop, scatter=False)
        if e2e:
            loss_host.copy_(state["loss"].reshape(1), non_blocking=True)   # the step's result read back
        done[i].record(cur)

    ms = timed(step, steps, D, warm=max(3, warmup))
    ms_e2e = timed(lambda k: step(k, True), steps, D, warm=2)
    ms, ms_e2e = D.max_ms(ms, ms_e2e)
    tflops = 3 * FLOP_PER_LR_PIXEL * B * (H // 4) * (W // 4) / (ms * 1e-3) / 1e12
    opt_info = None
    try:
        if not with_optimizer:
            raise RuntimeError("skipped")
        opt = resr_b200.optim.FlatAdamEMA(gen)
        flat = ts.flat
        for _ in range(2):
            opt.step(flat)
            gen._ensure_packed()
        torch.cuda.synchronize()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record()
        for _ in range(5):
            opt.step(flat)
            gen._ensure_packed()
        o1.record()
        torch.cuda.synchronize()
        opt_info = {"ms_per_step": o0.elapsed_time(o1) / 5,
                    "what": "resr_adam_ema_step (36 B per parameter) + repack of all tensor-core weight tiles (2 launches)"}
    except Exception as e:
        opt_info = None if not with_optimizer else {"error": repr(e)}
    return {"metric": "training pairs/s", "value": world * B / (ms * 1e-3), "unit": "pairs/s", "ms_per_step": ms, "n_gpus": world,
            "scaling": "weak", "loss": float(state["loss"].item()), "cuda_graph": bool(ts.is_graph), "optimizer": opt_info,
            "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "pairs/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": img_host.numel(), "d2h_bytes_per_step": 4,
                    "api": "per step: 16 decoded u8 HR images from pinned host memory -> DegradePipeline(u8_images=True) (augmentation + "
                           "degradation, one CUDA graph, on the data stream under the previous step) -> autograd.TrainStep.step; the loss "
                           "is read back to pinned host memory"},
            "precision": {"fp16": "fp16 activations, bf16 gradients, weight gradients through channels-first copies (wgrad_tc.cu)",
                          "bf16": "bf16 activations and gradients (north_star's recipe), fp32 residual stream, weight gradients "
                                  "straight from the NHWC buffers (wgrad_mn.cu)"}[precision],
            "config": {"workload": "per GPU and step: degradation (plan S0, mixed / sinc kernels, CUDA graph) of 16x3x256x256 HR + RRDBNet x4 "
                                   "forward/L1/backward on 16x3x64x64 LR (one CUDA graph), flat-gradient NCCL all-reduce (4 buckets under "
                                   "the backward) when n_gpus > 1; no optimizer. The degradation of batch k + 1 runs on a data stream "
                                   "under the training step of batch k"},
            "roofline": {"bound": "tensor", "achieved": tflops, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                         "frac": tflops / peaks["tf_sustained"], "traffic": None,
                         "note": "algorithmic FLOPs = 3 x forward (SURVEY.md §8d): 7.05 TFLOP per GPU-step"}}


# ------------------------------------------------------------------------------------------------- tiled inference (cfg5)


def tiled_bench(D, gen, steps, peaks):
    """configs[4]: 1x3x2048x2048 LR -> 1x3x8192x8192 SR. The image is cut into 8 full-width bands of 256 LR rows, each read
    with a 16-row halo (model.plan_tiles), dealt round-robin to the ranks; every rank uploads the LR image from pinned host
    memory, runs its bands, and the SR bands are gathered into rank 0's 8192^2 buffer with NCCL send / recv (contiguous row
    blocks, no staging copy); rank 0 copies the result to pinned host memory. All of it is inside the timer. Two variants:
    fp32 tensors in and out (what `model(lr_tensor)` returns, inference.py:53), and the u8 image path of inference.py:40-59
    (u8 image in, u8 image out: image_to_tensor / tensor_to_image fused into the first / last kernel, 4x fewer result bytes)."""
    import torch.distributed as dist

    import resr_b200
    device, world, rank = D.device, D.world, D.rank
    Hh = Ww = 2048
    tile_h, halo, s = 256, 16, 4
    g = torch.Generator(device="cpu").manual_seed(7)
    img_host = torch.randint(0, 256, (1, Hh, Ww, 3), generator=g, dtype=torch.uint8).pin_memory()      # decoded LR image (HWC u8)
    x_host = (img_host.permute(0, 3, 1, 2).float() / 255.0).contiguous().pin_memory()                  # the same image as a tensor
    tiles = resr_b200.model.plan_tiles(Hh, Ww, tile_h, Ww, halo)
    px = Hh * Ww
    halo_factor = sum((t[5] - t[4]) for t in tiles) / Hh

    def shared_host(shape, dtype, tag):
        """One result buffer in POSIX shared memory, mapped and page-locked (cudaHostRegister) by every rank: each rank's
        bands go device -> host over its OWN PCIe link straight into their rows of the one 8192^2 image."""
        import shutil
        numel = int(np.prod(shape))
        nbytes = numel * torch.empty((), dtype=dtype).element_size()
        base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > nbytes + (64 << 20) else "/tmp"
        path = f"{base}/resr_tiled_{os.environ.get('MASTER_PORT', '0')}_{tag}"
        def all_ok(ok):   # every rank learns whether every rank succeeded: nobody is left waiting in a barrier
            return D.max_ms(0.0 if ok else 1.0)[0] == 0.0

        ok = True
        if rank == 0:
            try:
                with open(path, "wb") as f:
                    f.truncate(nbytes)
            except OSError:
                ok = False
        if not all_ok(ok):
            raise RuntimeError(f"could not create {path}")
        t, ok = None, True
        try:
            t = torch.from_file(path, shared=True, size=numel, dtype=dtype).view(shape)
            ok = int(torch.cuda.cudart().cudaHostRegister(t.data_ptr(), nbytes, 0)) == 0
        except Exception:
            ok = False
        everyone = all_ok(ok)
        if rank == 0:
            try:
                os.unlink(path)   # the mappings keep the memory alive
            except OSError:
                pass
        if not everyone:
            if ok and t is not None:
                torch.cuda.cudart().cudaHostUnregister(t.data_ptr())
            raise RuntimeError("mapping / page-locking the shared result image failed on some rank")
        return t

    def run(u8, shared=False):
        tag = ("u8" if u8 else "f32")
        if u8:
            shape, dt = (1, s * Hh, s * Ww, 3), torch.uint8
            x_dev = torch.empty((1, Hh, Ww, 3), dtype=torch.uint8, device=device)
            src = img_host
        else:
            shape, dt = (1, 3, s * Hh, s * Ww), torch.float32
            x_dev = torch.empty((1, 3, Hh, Ww), dtype=torch.float32, device=device)
            src = x_host
        if shared:
            out, y_host = None, shared_host(shape, dt, tag)
        else:
            out = torch.empty(shape, dtype=dt, device=device) if rank == 0 else None
            y_host = torch.empty(shape, dtype=dt).pin_memory() if rank == 0 else None

        def step(k):
            if shared:   # only the windows this rank computes are uploaded
                for i, (y0, y1, x0, x1, wy0, wy1, wx0, wx1) in enumerate(tiles):
                    if i % world == rank:
                        if u8:
                            x_dev[:, wy0:wy1].copy_(src[:, wy0:wy1], non_blocking=True)
                        else:
                            x_dev[:, :, wy0:wy1].copy_(src[:, :, wy0:wy1], non_blocking=True)
            else:
                x_dev.copy_(src, non_blocking=True)
            ops, keep = [], []
            for i, (y0, y1, x0, x1, wy0, wy1, wx0, wx1) in enumerate(tiles):
                owner = i % world
                r0, r1 = s * (y0 - wy0), s * (y0 - wy0) + s * (y1 - y0)
                if owner == rank:
                    if u8:
                        piece = gen.infer_u8(x_dev[:, wy0:wy1])[:, r0:r1]               # [1, rows, 4W, 3]: one contiguous block
                        parts = [(piece[0], (y_host if shared else out)[0, s * y0:s * y1] if (shared or rank == 0) else None)]
                    else:
                        sr = gen.infer(x_dev[:, :, wy0:wy1, :])
                        parts = [(sr[0, c, r0:r1], (y_host if shared else out)[0, c, s * y0:s * y1] if (shared or rank == 0) else None)
                                 for c in range(3)]
                    for piece_c, dst in parts:
                        if shared:
                            dst.copy_(piece_c, non_blocking=True)   # D2H of this rank's rows into the shared pinned image
                            keep.append(piece_c)
                        elif rank == 0:
                            dst.copy_(piece_c)
                        else:
                            t = piece_c.contiguous()
                            keep.append(t)
                            ops.append(dist.P2POp(dist.isend, t, 0))
                elif rank == 0 and not shared:
                    dsts = [out[0, s * y0:s * y1]] if u8 else [out[0, c, s * y0:s * y1] for c in range(3)]
                    for dst in dsts:
                        ops.append(dist.P2POp(dist.irecv, dst, owner))
            if ops:
                for w in dist.batch_isend_irecv(ops):
                    w.wait()
            if rank == 0 and not shared:
                y_host.copy_(out, non_blocking=True)
            if shared:
                torch.cuda.current_stream(device).synchronize()   # `keep` may go: this rank's copies have landed

        ms = timed(step, steps, D, warm=1)
        ms = D.max_ms(ms)[0]
        chk = None
        if rank == 0:
            chk = float(y_host[0, ::512, ::512].double().sum()) if u8 else float(y_host[0, :, ::512, ::512].double().sum())
        if shared:
            D.barrier()
            torch.cuda.cudart().cudaHostUnregister(y_host.data_ptr())
        nbytes_in = src.numel() * src.element_size()
        nbytes_out = 3 * 16 * px * (1 if u8 else 4)
        if shared:
            return {"value": px / (ms * 1e-3) / 1e6, "unit": "LR Mpix/s", "ms_per_step": ms,
                    "h2d_bytes_per_step": int(nbytes_in * halo_factor), "d2h_bytes_per_step": nbytes_out, "gather_bytes_per_step": 0,
                    "checksum": chk}
        return {"value": px / (ms * 1e-3) / 1e6, "unit": "LR Mpix/s", "ms_per_step": ms, "h2d_bytes_per_step": nbytes_in * world,
                "d2h_bytes_per_step": nbytes_out, "gather_bytes_per_step": nbytes_out * (world - 1) // world, "checksum": chk}

    f32 = run(False)
    gen._workspace = None
    torch.cuda.empty_cache()
    u8 = run(True)
    sh = {}
    for name, is_u8 in (("fp32", False), ("u8_image", True)):
        gen._workspace = None
        torch.cuda.empty_cache()
        try:
            sh[name] = run(is_u8, shared=True)
        except Exception as e:   # e.g. no /dev/shm: keep the NCCL-gather numbers
            sh[name] = {"error": repr(e)}
        if "checksum" in sh[name] and rank == 0:
            ref = (u8 if is_u8 else f32)["checksum"]
            sh[name]["matches_nccl_gather"] = bool(sh[name]["checksum"] == ref)
    # headline of the leg: the faster of the two ways of assembling the fp32 result in ONE pinned host buffer
    best, how = f32, "NCCL send/recv gather into rank 0's buffer, then one device -> host copy"
    if sh["fp32"].get("matches_nccl_gather") or (world > 1 and rank != 0):
        if sh["fp32"].get("ms_per_step", float("inf")) < f32["ms_per_step"]:
            best, how = sh["fp32"], "no gather: every rank copies its bands into one page-locked host image in shared memory"
    ms = best["ms_per_step"]
    tflops = FLOP_PER_LR_PIXEL * px * halo_factor / (ms * 1e-3) / 1e12
    tflops8 = FLOP_PER_LR_PIXEL * px * halo_factor / (u8["ms_per_step"] * 1e-3) / 1e12
    return {"metric": "tiled x4 inference LR Mpix/s", "value": best["value"], "unit": "LR Mpix/s", "ms_per_step": ms,
            "n_gpus": world, "scaling": "strong", "steps": steps,
            "config": {"workload": "1x3x2048x2048 LR -> 1x3x8192x8192 SR (BASELINE.json configs[4]), 8 full-width bands of 256 LR rows "
                                   f"+ 16-row halo ({halo_factor:.3f}x pixels computed), round-robin over {world} rank(s); timed end to "
                                   f"end from / to pinned host memory (fp32 tensors); result assembled by: {how}"},
            "e2e": best,
            "nccl_gather": f32,
            "shared_pinned_host": dict(sh, api="no gather at all: the result image lives in ONE page-locked host buffer in POSIX shared "
                                               "memory mapped by every rank (cudaHostRegister); each rank uploads only its windows and "
                                               "copies its bands device -> host over its own PCIe link into their rows (SURVEY.md §8e: "
                                               "'gather by P2P copy into one GPU's buffer or pinned host')"),
            "u8_image": dict(u8, api="Generator.infer_u8 per band (resr_generator_forward_u8): u8 HWC image in, u8 HWC image out, the "
                                     "conversions of inference.py:40-46, 56 fused into the first / last kernel",
                             roofline_frac=tflops8 / (peaks["tf_sustained"] * world)),
            "roofline": {"bound": "tensor", "achieved": tflops, "peak": peaks["tf_sustained"] * world, "unit": "TFLOP/s",
                         "frac": tflops / (peaks["tf_sustained"] * world),
                         "note": "halo pixels counted as work; copies and gather are inside the time"}}


# ------------------------------------------------------------------------------------------------- arms


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import generator as og
    torch.set_num_threads(os.cpu_count() or 1)
    sd = og.random_state_dict(0)
    torch.manual_seed(0)
    x = torch.rand(1, 3, 128, 128)
    for _ in range(max(1, min(args.warmup, 2))):
        og.generator_forward(x, sd)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        y = og.generator_forward(x, sd)
    dt = (time.perf_counter() - t0) / args.steps
    val = 128 * 128 / dt / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "LR Mpix/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "RRDBNet x4 (23 RRDB, nf=64, gc=32) forward, random init; each step a bounded sample "
                                   "of the 64x3x128x128 workload: one 1x3x128x128 image on the host CPU"},
            "cpu_baseline": {"value": val, "unit": "LR Mpix/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": "1x3x128x128 fp32 forward per step, oracle port of model.py (reference tree is not on the GPU box)"},
            "e2e": {"value": val, "unit": "LR Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if args.dump_outputs:
        line["dump_outputs"] = dump_output(args.dump_outputs, "sr", y)
    try:  # secondary: the degradation half of the metric on the same host cores (numpy port, bounded sample)
        import resr_b200
        from oracle import kernels as ok
        P = resr_b200.plan.DEGRADATION_MODEL_PARAMETERS
        random.seed(0)
        np.random.seed(0)
        ks = []
        for _ in range(4):
            p, _ = resr_b200.imgproc.draw_mixed_kernel_params(P["gaussian_kernel_type"], P["gaussian_kernel_probability1"], 21,
                                                              P["gaussian_sigma_range1"], P["gaussian_sigma_range1"], [-math.pi, math.pi],
                                                              P["generalized_kernel_beta_range1"], P["plateau_kernel_beta_range1"])
            ks.append(ok.from_params(p, 21))
        k = np.stack(ks).astype(np.float32)
        sk = np.stack([ok.from_params({"type": "sinc", "kernel_size": 21, "cutoff": 2.0}, 21)] * 4).astype(np.float32)
        line["degradation"] = cpu_degradation_baseline((k, k, sk))
    except Exception as e:
        line["degradation"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)


def run_ours(args):
    D = Dist()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA (B200) device: there is no CPU fallback for the product path")
    D.init()
    world, rank, device = D.world, D.rank, D.device
    import resr_b200
    L = resr_b200._lib
    peaks = measured_peaks()
    torch.set_grad_enabled(False)

    H = W = 128
    if args.batch:
        n_strong = args.batch
    else:
        n_strong = max(1, TOTAL_BATCH // world)   # strong scaling: the 64 images of configs[2] sharded over the ranks
    torch.manual_seed(0)
    gen = resr_b200.model.Generator(3, 3, 4).to(device).eval()
    if args.precision != "fp16":
        gen.set_precision(args.precision)
    gen.assume_static_weights(True)
    launches = L.lib().resr_generator_launches_per_forward()

    def forward_leg(n):
        gcpu = torch.Generator().manual_seed(1234 + rank)
        x_host = torch.rand(n, 3, H, W, generator=gcpu).pin_memory()
        y_hosts = [torch.empty(n, 3, 4 * H, 4 * W).pin_memory() for _ in range(2)]
        x = x_host.to(device)
        state = {}

        def dev_step(k):
            state["y"] = gen(x)

        with ClockSampler(D.local) as clocks:
            ms = timed(dev_step, args.steps, D, warm=max(3, args.warmup))
        e2e_steps = max(4, min(args.steps, 10))
        ms_block = timed(lambda k: gen.infer_host(x_host, y_hosts[0], device), e2e_steps, D, warm=2)
        ms_pipe = timed(lambda k: gen.infer_host_async(x_host, y_hosts[k & 1], device), e2e_steps, D, fin=gen.host_sync, warm=2)
        ms, ms_block, ms_pipe = D.max_ms(ms, ms_block, ms_pipe)
        return {"n": n, "ms": ms, "ms_block": ms_block, "ms_pipe": ms_pipe, "clocks": clocks.summary(),
                "h2d": x_host.numel() * 4, "d2h": y_hosts[0].numel() * 4,
                "checksum": float(y_hosts[0][0, :, ::64, ::64].double().sum()), "y": state["y"]}

    head = forward_leg(n_strong)
    dumped = dump_output(args.dump_outputs, "sr", head["y"]) if args.dump_outputs and rank == 0 else None
    head["y"] = None
    weak = forward_leg(TOTAL_BATCH) if (world > 1 and not args.batch and not args.no_weak) else None
    # the other precision recipe on the same box, device-resident only (north_star names bf16; fp16 is the default)
    other = "bf16" if args.precision == "fp16" else "fp16"
    other_ms = None
    if not args.no_other_precision:
        try:
            gen.set_precision(other)
            gen.invalidate()
            xo = torch.rand(n_strong, 3, H, W, generator=torch.Generator().manual_seed(99 + rank)).to(device)
            other_ms = D.max_ms(timed(lambda k: gen(xo), max(3, args.steps // 2), D, warm=3))[0]
        finally:
            gen.set_precision(args.precision)
            gen.invalidate()
            gen._workspace = None

    line = None
    if rank == 0:
        px = world * head["n"] * H * W
        tflops = FLOP_PER_LR_PIXEL * px / (head["ms"] * 1e-3) / 1e12
        prec = {"fp16": "fp16 MMA operands (16-bit tensor-core rate, same as bf16), fp32 accumulate and fp32 epilogue arithmetic; the "
                        "trunk residual stream is the fp16 conv input (saturating at 65504)",
                "bf16": "bf16 MMA operands and stored activations, fp32 accumulate, fp32 residual masters for the trunk (north_star recipe)"}
        line = {
            "metric": METRIC, "value": px / (head["ms"] * 1e-3) / 1e6, "unit": "LR Mpix/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": head["ms"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": {"workload": f"RRDBNet x4 (23 RRDB, nf=64, gc=32) inference, {world * head['n']}x3x{H}x{W} LR in total "
                                   f"(BASELINE.json configs[2]), {head['n']} images per GPU, random init; batch-sharded, no collective",
                       "precision": prec[args.precision],
                       "other_precision": None if other_ms is None else {
                           "recipe": other, "what": prec[other], "value": px / (other_ms * 1e-3) / 1e6, "unit": "LR Mpix/s",
                           "ms_per_step": other_ms,
                           "roofline_frac": FLOP_PER_LR_PIXEL * px / (other_ms * 1e-3) / 1e12 / (peaks["tf_sustained"] * world)},
                       "l2": "working set (GBs of activations per forward) is far larger than the 126 MB L2; no flush needed"},
            "e2e": {"value": px / (head["ms_pipe"] * 1e-3) / 1e6, "unit": "LR Mpix/s", "ms_per_step": head["ms_pipe"],
                    "h2d_bytes_per_step": head["h2d"], "d2h_bytes_per_step": head["d2h"],
                    "api": "resr_generator_forward_host_async + resr_generator_host_sync (pinned host buffers, pipelined)",
                    "blocking_call": {"value": px / (head["ms_block"] * 1e-3) / 1e6, "ms_per_step": head["ms_block"],
                                      "api": "resr_generator_forward_host"},
                    "checksum": head["checksum"]},
            "gpu_launches": launches * args.steps,
            "clocks": head["clocks"],
            "roofline": {"bound": "tensor", "achieved": tflops, "peak": peaks["tf_sustained"] * world, "unit": "TFLOP/s",
                         "frac": tflops / (peaks["tf_sustained"] * world),
                         # dram__bytes_read.sum + dram__bytes_write.sum per launch, mean over the launches of one forward at cfg3
                         # (ncu capture under profiles/, see profiles/README.md)
                         "traffic": TRAFFIC_PER_LAUNCH if (head["n"], world) == (64, 1) else None,
                         "kernel": "conv3x3_pair_kernel (tcgen05 cta_group::2; 351 conv launches per forward; algorithmic FLOPs "
                                   "35,853,696 per LR pixel)",
                         "peak_source": peaks["source"] + " bf16_tflops_sustained (kernel timed inside a long step), x n_gpus"},
        }
        if dumped is not None:
            line["dump_outputs"] = dumped
        if weak is not None:
            wpx = world * weak["n"] * H * W
            line["weak"] = {"value": wpx / (weak["ms"] * 1e-3) / 1e6, "unit": "LR Mpix/s", "ms_per_step": weak["ms"],
                            "images_per_gpu": weak["n"], "e2e": wpx / (weak["ms_pipe"] * 1e-3) / 1e6,
                            "roofline_frac": FLOP_PER_LR_PIXEL * wpx / (weak["ms"] * 1e-3) / 1e12 / (peaks["tf_sustained"] * world)}

    # ---- configs[4]: tiled large-image inference over the ranks, with the gather
    tiled = None
    if not args.no_tiled:
        try:
            tiled = tiled_bench(D, gen, 2 if world == 1 else 3, peaks)
        except Exception as e:
            tiled = {"error": repr(e)}
            D.barrier()
    gen._workspace = None   # the 2048-wide bands held ~20 GB of activations
    torch.cuda.empty_cache()

    # ---- configs[1]: degradation; every rank degrades its own batches (no collective on the path)
    deg = None
    if not args.no_degrade:
        err, r16, r256 = None, None, None
        try:
            r16 = degradation_bench(D, max(20, args.steps), args.warmup, peaks, B=16)
            r256 = degradation_bench(D, 10, 3, peaks, B=256, want_e2e=False)  # large-batch regime (SURVEY.md §8d)
        except Exception as e:  # keep the headline even if the secondary leg breaks
            err = repr(e)
        vals = D.max_ms(*( [r16["ms_dev"], r16["ms_e2e"], r256["ms_dev"], r16["ms_e2e_u8"]] if err is None else [float("inf")] * 4))
        if rank == 0:
            if err is not None or vals[0] == float("inf"):
                deg = {"error": err or "another rank failed"}
            else:
                m16, me2e, m256, me2e_u8 = vals
                sbytes, stages, _ = s0_stage_bytes(16)
                gbs = sbytes / (m16 * 1e-3) / 1e9
                tfma = r16["fma"] / (m16 * 1e-3) / 1e12
                deg = {"metric": "degraded pairs/s", "value": world * 16 / (m16 * 1e-3), "unit": "pairs/s", "ms_per_step": m16,
                       "n_gpus": world, "scaling": "weak",
                       "config": {"workload": "second-order degradation, 16x3x256x256 HR -> 16x3x64x64 LR per GPU, canonical plan S0 "
                                              "(SURVEY.md §8d) with mixed Gaussian-family / sinc blur kernels of support 7..21 and a real "
                                              "sinc final kernel; Gaussian noise tensors host-fed and resident, Poisson draws made inside "
                                              "the fused noise kernel (Philox); one CUDA-graph replay per batch"},
                       "e2e": {"value": world * 16 / (me2e * 1e-3), "unit": "pairs/s", "ms_per_step": me2e,
                               "h2d_bytes_per_step": r16["h2d"], "d2h_bytes_per_step": r16["d2h"],
                               "api": "imgproc.DegradePipeline x 2 (alternating CUDA graphs): HR batch from pinned host memory every "
                                      "step, LR batch read back to pinned host memory; HR crop stays on the device for the training step"},
                       "e2e_u8_images": {"value": world * 16 / (me2e_u8 * 1e-3), "unit": "pairs/s", "ms_per_step": me2e_u8,
                                         "h2d_bytes_per_step": r16["h2d_u8"], "d2h_bytes_per_step": r16["d2h"],
                                         "api": "the same, but the batch arrives as decoded u8 HWC BGR images (cv2.imread's output, "
                                                "dataset.py:67): / 255 + rotate / flips + BGR->RGB + HWC->CHW of dataset.py:67-79 run as "
                                                "imgproc.augment_batch (one gather kernel, the first node of the pipeline's CUDA graph)"},
                       "gpu_launches_per_step": DEGRADE_LAUNCHES,
                       "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"],
                                    "traffic": DEGRADE_TRAFFIC, "algorithmic_bytes_per_step": sbytes,
                                    "note": "stage-sum bytes / whole-pipeline time, per GPU; the blur stencils are fp32-FMA work: see fma"},
                       "fma": {"achieved_tfma": tfma, "peak_tfma": peaks["tfma"], "frac": tfma / peaks["tfma"],
                               "necessary_fma_per_step": r16["fma"],
                               "note": "necessary FMAs (separable 51-tap USM, per-sample trimmed blur supports) / whole-pipeline time vs the "
                                       "fp32 FMA peak measured with tools/fma_peak.cu (profiles/r02_fma_peak.json)"},
                       "large_batch": {"batch_per_gpu": 256, "value": world * 256 / (m256 * 1e-3), "unit": "pairs/s", "ms_per_step": m256,
                                       "roofline_frac": s0_stage_bytes(256)[0] / (m256 * 1e-3) / 1e9 / peaks["hbm"]}}
                if world == 1 and not args.no_cpu:
                    try:
                        deg["cpu_baseline"] = cpu_degradation_baseline(r16["kernels_np"])
                    except Exception as e:
                        deg["cpu_baseline"] = {"error": repr(e)}
    if rank == 0:
        if tiled is not None:
            line["tiled"] = tiled
        if deg is not None:
            line["degradation"] = deg
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_generator_baseline()
    train = None
    if not args.no_train:  # every rank takes part (all-reduce)
        try:
            train = training_bench(D, max(5, min(args.steps, 20)), args.warmup, peaks, args.train_precision)
            if not args.no_other_precision:
                other_t = "fp16" if args.train_precision == "bf16" else "bf16"
                try:
                    o = training_bench(D, max(5, min(args.steps, 10)), args.warmup, peaks, other_t, with_optimizer=False)
                    train["other_precision"] = {"recipe": other_t, "what": o["precision"], "value": o["value"], "unit": o["unit"],
                                                "ms_per_step": o["ms_per_step"], "loss": o["loss"]}
                except Exception as e:
                    train["other_precision"] = {"recipe": other_t, "error": repr(e)}
        except Exception as e:
            train = {"error": repr(e)}
    if rank == 0:
        line["training"] = train
        print(json.dumps(line), flush=True)
    D.finish()


# ncu-measured DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum), see profiles/README.md for the captures
TRAFFIC_PER_LAUNCH = 380.2e6   # bytes per conv launch, mean over the 351 launches of one cfg3 forward (profiles/r02_generator_launches_v2.csv)
DEGRADE_TRAFFIC = 133.6e6      # bytes per S0 batch, sum over the 15 launches, cold L2 (profiles/r02_degrade_launches_v2.csv)
DEGRADE_LAUNCHES = 15


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, metavar="K",
                    help="timed steps of the headline leg (the one --dump-outputs writes); the secondary legs clamp it to "
                         "their own counts: e2e max(4, min(K, 10)), other precision max(3, K // 2), degradation max(20, K) "
                         "(large batch: 10), training max(5, min(K, 20)) (other precision: max(5, min(K, 10))), tiled 2 "
                         "(3 for N > 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16"],
                    help="MMA operand / activation format of the generator (bf16 = north_star's recipe with fp32 residual masters)")
    ap.add_argument("--batch", type=int, default=0, help="LR images per GPU (default 64 / n_gpus: strong scaling of configs[2])")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--train-precision", choices=["fp16", "bf16"], default="bf16",
                    help="recipe of the training leg (bf16: north_star's recipe, NHWC weight-gradient kernel)")
    ap.add_argument("--no-other-precision", action="store_true", help="skip the secondary forward leg in the other precision recipe")
    ap.add_argument("--no-weak", action="store_true", help="skip the secondary weak-scaling forward leg (N > 1)")
    ap.add_argument("--no-tiled", action="store_true", help="skip the secondary tiled-inference leg (configs[4])")
    ap.add_argument("--no-degrade", action="store_true", help="skip the secondary degradation leg")
    ap.add_argument("--no-train", action="store_true", help="skip the secondary training-step leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the SR batch of the last timed step to DIR/sr.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
