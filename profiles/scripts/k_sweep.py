"""BASELINE config 4 on one GPU: diff-drive K = 1M..64M, H = 50 (sum/frozen, Philox), device-timed ticks."""
import os, sys; sys.path[:0] = [os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]
import numpy as np, torch
from bench import diffdrive_kwargs
from mppi_b200.mppi_differential_drive import MPPIAlgorithms
for K in (1 << 20, 1 << 22, 1 << 24, 1 << 26):
    c = MPPIAlgorithms(**diffdrive_kwargs(K, 50, 10.0), seed=7)
    eng = c.engine
    st = torch.cuda.Stream(); eng.set_stream(st.cuda_stream)
    for i in range(3): eng.step_async(np.zeros(3), None, 7, i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = max(3, (1 << 25) // K)
    a.record(st)
    for i in range(n): eng.step_async(np.zeros(3), None, 7, 10 + i)
    b.record(st); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / n
    s = eng.stats()
    print(f"K={K:>9d} H=50: {ms:9.3f} ms/tick  {K*50/ms/1e6:8.2f} G sample-steps/s  ess={s['ess']:.0f} eta={s['eta']:.4g}", flush=True)
    eng.set_stream(0); eng.close()
