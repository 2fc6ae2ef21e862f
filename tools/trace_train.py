"""Kernel timeline of one training step via torch.profiler (CUPTI): do the data-gradient and weight-gradient chains overlap?"""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from torch.profiler import profile, ProfilerActivity
import resr_b200
n, h, w = 16, 64, 64
torch.manual_seed(0)
g = resr_b200.model.Generator(3, 3, 4).cuda().train()
g.set_precision(os.environ.get("RESR_PREC", "bf16"))
lr = torch.rand(n, 3, h, w, device="cuda"); hr = torch.rand(n, 3, 4 * h, 4 * w, device="cuda")
ts = resr_b200.autograd.TrainStep(g, n, h, w)
for _ in range(3):
    ts.step(lr, hr, scatter=False)
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    ts.step(lr, hr, scatter=False)
    torch.cuda.synchronize()
prof.export_chrome_trace("/tmp/train_trace.json")
ev = [e for e in json.load(open("/tmp/train_trace.json"))["traceEvents"] if e.get("cat") == "kernel"]
ev.sort(key=lambda e: e["ts"])
print("kernels", len(ev), "span ms", (ev[-1]["ts"] + ev[-1]["dur"] - ev[0]["ts"]) / 1e3, "sum ms", sum(e["dur"] for e in ev) / 1e3)
streams = sorted(set(e["args"].get("stream") for e in ev))
print("streams", streams)
# overlap between conv kernels and wgrad kernels
import bisect
conv = [(e["ts"], e["ts"] + e["dur"]) for e in ev if "conv3x3" in e["name"]]
wg = [(e["ts"], e["ts"] + e["dur"]) for e in ev if "wgrad_mn_kernel" in e["name"]]
ov = 0.0
for a0, a1 in wg:
    for b0, b1 in conv:
        if b0 >= a1: break
        if b1 <= a0: continue
        ov += min(a1, b1) - max(a0, b0)
print(f"wgrad total {sum(b-a for a,b in wg)/1e3:.2f} ms, conv total {sum(b-a for a,b in conv)/1e3:.2f} ms, overlapped {ov/1e3:.2f} ms")
# print a window of the backward timeline
mid = len(ev) // 2
t0 = ev[mid]["ts"]
for e in ev[mid:mid + 24]:
    print(f"{e['ts']-t0:9.1f} +{e['dur']:6.1f} us  stream {e['args'].get('stream')}  {e['name'][:40]}  grid {e['args'].get('grid')}")
# per-kernel-name totals and the time span of forward / backward phases
import collections
tot = collections.Counter()
cnt = collections.Counter()
for e in ev:
    nm = e["name"].split("(")[0].split("<")[0][-36:]
    tot[nm] += e["dur"]
    cnt[nm] += 1
for nm, d in tot.most_common(14):
    print(f"  {nm:38s} n={cnt[nm]:5d} total {d/1e3:7.2f} ms  mean {d/cnt[nm]:6.1f} us")
by_stream = collections.Counter()
for e in ev:
    by_stream[e["args"].get("stream")] += e["dur"]
print("busy per stream (ms):", {k: round(v / 1e3, 2) for k, v in by_stream.items()})
first_bwd = next(i for i, e in enumerate(ev) if "out_grad" in e["name"])
print(f"forward span {(ev[first_bwd]['ts'] - ev[0]['ts'])/1e3:.2f} ms, backward span {(ev[-1]['ts'] + ev[-1]['dur'] - ev[first_bwd]['ts'])/1e3:.2f} ms")
