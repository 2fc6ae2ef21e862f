"""Quick device-timed forward of the generator (development aid; bench.py is the contract)."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import resr_b200
torch.set_grad_enabled(False)

n, h, w = (int(v) for v in (sys.argv[1:4] if len(sys.argv) >= 4 else (64, 128, 128)))
torch.manual_seed(0)
g = resr_b200.model.Generator(3, 3, 4).cuda().eval()
x = torch.rand(n, 3, h, w, device="cuda")
for _ in range(2):
    y = g(x)
torch.cuda.synchronize()
ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
iters = 5
ev0.record()
for _ in range(iters):
    y = g(x)
ev1.record()
torch.cuda.synchronize()
ms = ev0.elapsed_time(ev1) / iters
flop = 35853696.0 * n * h * w
print(f"{n}x3x{h}x{w}: {ms:.3f} ms/forward  {n*h*w/ms/1e3:.3f} LR Mpix/s  {flop/ms/1e9:.1f} TFLOP/s")
