"""Where the ~8 us between the back-to-back tick time and bench.py's per-step event time come from: per-step CUDA events with
(a) nothing, (b) the 256 MiB L2-flush memset, (c) a small unrelated kernel between the ticks."""
import os, sys; sys.path[:0]=[os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]
import numpy as np, torch
from bench import diffdrive_kwargs
from mppi_b200.mppi_differential_drive import MPPIAlgorithms
c = MPPIAlgorithms(**diffdrive_kwargs(1 << 20, 50, 10.0), seed=7)
eng = c.engine
st = torch.cuda.Stream(); eng.set_stream(st.cuda_stream)
x0 = np.zeros(3)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
small = torch.empty(1 << 16, dtype=torch.float32, device="cuda")
for i in range(10): eng.step_async(x0, None, 7, i)
torch.cuda.synchronize()
def run(mode, n=60):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    with torch.cuda.stream(st):
        for i in range(n):
            if mode == "flush": flush.zero_()
            elif mode == "small": small.zero_()
            ev[i][0].record(st); eng.step_async(x0, None, 7, 100 + i); ev[i][1].record(st)
    torch.cuda.synchronize()
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    return ms.mean(), np.median(ms)
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record(st)
for i in range(60): eng.step_async(x0, None, 7, 50 + i)
b.record(st); torch.cuda.synchronize()
print("back to back, one event pair around 60 ticks: %.4f ms/tick" % (a.elapsed_time(b) / 60))
for mode in ("none", "small", "flush", "none", "flush"):
    print("per-step events, between ticks = %-5s: mean %.4f median %.4f ms" % ((mode,) + run(mode)))
