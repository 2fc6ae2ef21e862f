"""Sustained forward loop with NVML power / clock sampling (development aid)."""
import sys, os, time, threading
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, pynvml
import resr_b200
torch.set_grad_enabled(False)
n, h, w = 64, 128, 128
secs = float(sys.argv[1]) if len(sys.argv) > 1 else 4.0
g = resr_b200.model.Generator(3, 3, 4).cuda().eval()
x = torch.rand(n, 3, h, w, device="cuda")
for _ in range(2):
    g(x)
torch.cuda.synchronize()
pynvml.nvmlInit()
hd = pynvml.nvmlDeviceGetHandleByIndex(0)
rows, stop = [], threading.Event()
def run():
    while not stop.is_set():
        rows.append((pynvml.nvmlDeviceGetPowerUsage(hd) / 1e3, pynvml.nvmlDeviceGetClockInfo(hd, pynvml.NVML_CLOCK_SM),
                     pynvml.nvmlDeviceGetClockInfo(hd, pynvml.NVML_CLOCK_MEM)))
        stop.wait(0.02)
t = threading.Thread(target=run, daemon=True); t.start()
t0 = time.time(); times = []
while time.time() - t0 < secs:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        g(x)
    e1.record(); torch.cuda.synchronize()
    times.append(e0.elapsed_time(e1) / 5)
stop.set(); t.join()
half = rows[len(rows) // 2:]
med = lambda v: sorted(v)[len(v) // 2]
print(f"first {times[0]:.2f} ms  last {times[-1]:.2f} ms  "
      f"power {med([r[0] for r in half]):.0f} W  sm {med([r[1] for r in half])} MHz  mem {med([r[2] for r in half])} MHz  "
      f"limit {pynvml.nvmlDeviceGetEnforcedPowerLimit(hd)/1e3:.0f} W")
