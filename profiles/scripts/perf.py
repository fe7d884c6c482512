import os, sys, time; sys.path[:0]=[os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]
import numpy as np, torch
from bench import diffdrive_kwargs
from mppi_b200.mppi_differential_drive import MPPIAlgorithms
from mppi_b200.mppi_race_car_obstacle import MPPIRacecarController
def timeit(eng, x0, n=30):
    st = torch.cuda.Stream(); eng.set_stream(st.cuda_stream)
    for i in range(5): eng.step_async(x0, None, 7, i)
    torch.cuda.synchronize()
    a,b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for i in range(n): eng.step_async(x0, None, 7, 10+i)
    b.record(st); torch.cuda.synchronize()
    return a.elapsed_time(b)/n
for K,T,temp in ((1<<20,50,10.0),(1<<20,50,None),(1<<22,50,10.0)):
    c = MPPIAlgorithms(**diffdrive_kwargs(K,T,temp), seed=7)
    ms = timeit(c.engine, np.zeros(3))
    print(f"diffdrive K={K} T={T} temp={temp}: {ms:.4f} ms  {K*T/ms/1e6:.2f} G sample-steps/s", flush=True)
    c.engine.close()
rc = MPPIRacecarController(horizon_step_T=50, number_of_samples_K=16384, visualize_optimal_traj=False, visualze_sampled_trajs=False, seed=3)
lp = rc.generate_lemniscate_trajectory(100, 10.0).astype(np.float32); rc.ref_path = lp
ms = timeit(rc.engine, lp[0].astype(np.float64), 100)
print(f"racecar K=16384 T=50 device: {ms*1e3:.1f} us/tick")
rc.engine.set_stream(0)
lat=[]
for i in range(300):
    rc.prev_waypoints_idx = 0
    t=time.perf_counter(); rc._calc_control_input(lp[i%50]); lat.append(time.perf_counter()-t)
lat=np.sort(lat); print(f"racecar host p50 {lat[150]*1e6:.1f} us p90 {lat[270]*1e6:.1f} us")
rc.engine.close()
rc = MPPIRacecarController(horizon_step_T=50, number_of_samples_K=1<<20, visualize_optimal_traj=False, visualze_sampled_trajs=False, seed=3)
rc.ref_path = lp
ms = timeit(rc.engine, lp[0].astype(np.float64), 10)
print(f"racecar K=1M T=50: {ms:.3f} ms {(1<<20)*50/ms/1e6:.2f} G sample-steps/s")
