import sys, time, os; sys.path[:0]=[os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]
import numpy as np, torch
from mppi_b200.mppi_race_car_obstacle import MPPIRacecarController
from mppi_b200.mppi_differential_drive import MPPIAlgorithms
from bench import diffdrive_kwargs
def timeit(eng, x0, n=200):
    st = torch.cuda.Stream(); eng.set_stream(st.cuda_stream)
    for i in range(20): eng.step_async(x0, None, 7, i)
    torch.cuda.synchronize()
    a,b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for i in range(n): eng.step_async(x0, None, 7, 30+i)
    b.record(st); torch.cuda.synchronize()
    eng.set_stream(0)
    return a.elapsed_time(b)/n
print("MIN_CTA", os.environ.get("MPPI_MIN_CTA_SAMPLES"))
for K in (1024, 4096, 16384, 65536, 262144):
    rc = MPPIRacecarController(horizon_step_T=50, number_of_samples_K=K, visualize_optimal_traj=False, visualze_sampled_trajs=False, seed=3)
    lp = rc.generate_lemniscate_trajectory(100, 10.0).astype(np.float32); rc.ref_path = lp
    ms = timeit(rc.engine, lp[0].astype(np.float64))
    lat=[]
    for i in range(300):
        rc.prev_waypoints_idx = 0
        t=time.perf_counter(); rc._calc_control_input(lp[i%50]); lat.append(time.perf_counter()-t)
    lat=np.sort(lat)
    print(f"racecar K={K}: device {ms*1e3:.1f} us/tick; host p50 {lat[150]*1e6:.1f} us", flush=True)
    rc.engine.close()
for K in (1000, 16384, 65536):
    c = MPPIAlgorithms(**diffdrive_kwargs(K,30,10.0), seed=7)
    ms = timeit(c.engine, np.zeros(3))
    print(f"diffdrive K={K} T=30: device {ms*1e3:.1f} us/tick", flush=True)
    c.engine.close()
