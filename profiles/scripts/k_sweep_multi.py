"""BASELINE config 5 under torchrun: diff-drive, H = 50 (sum/frozen, Philox), K_global = 16M / 64M sharded over the ranks of
one box, fused NVLink exchange, device-timed per tick (CUDA events on the launching stream), MAX over ranks.
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P profiles/scripts/k_sweep_multi.py"""
import os, sys
sys.path[:0] = [os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]
import numpy as np, torch, torch.distributed as dist
from bench import diffdrive_kwargs
from mppi_b200.mppi_differential_drive import MPPIAlgorithms
rank, world, lr = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(lr)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
for Kg in (1 << 24, 1 << 26):
    c = MPPIAlgorithms(**diffdrive_kwargs(Kg, 50, 10.0), seed=7, device=lr, rank=rank, world=world)
    if world > 1:
        c.comm_init_from_torch()
    eng = c.engine
    st = torch.cuda.Stream(); eng.set_stream(st.cuda_stream)
    for i in range(3): eng.step_async(np.zeros(3), None, 7, i)
    torch.cuda.synchronize()
    if world > 1: dist.barrier()
    n = 10
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    with torch.cuda.stream(st):
        for i in range(n):
            ev[i][0].record(st); eng.step_async(np.zeros(3), None, 7, 10 + i); ev[i][1].record(st)
    torch.cuda.synchronize()
    t = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], device="cuda", dtype=torch.float64)
    if world > 1: dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / n
    if rank == 0:
        print(f"GPUs={world} K_global={Kg:>9d} (K/GPU={Kg // world}) H=50: {ms:8.3f} ms/tick  {Kg * 50 / ms / 1e6:9.2f} G sample-steps/s", flush=True)
    eng.set_stream(0); eng.close()
if world > 1:
    dist.destroy_process_group()
