"""Where the literal C1 tick (K = 1000, T = 30, cost_mode last, waypoint_mode strict) spends its time: the handle's own event
timings (rollout = strict passes incl. their host round trips, update = K2 kernel) next to the host-to-host latency."""
import sys, time
import os
sys.path[:0] = [os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]
import numpy as np
from bench import diffdrive_kwargs
from mppi_b200.mppi_differential_drive import MPPIAlgorithms
kw = diffdrive_kwargs(1000, 30, None)
kw.update(cost_mode="last", waypoint_mode="strict", param_exploration=0.05)
c = MPPIAlgorithms(**kw, seed=7)
x = np.zeros(3)
for i in range(30):
    c._calc_input_control(x)
lat = []
for i in range(200):
    t = time.perf_counter(); c._calc_input_control(x); lat.append(time.perf_counter() - t)
print("host p50 %.1f us (no timing events)" % (1e6 * np.median(lat)))
c.engine.set_timing(True)
rows = []
for i in range(200):
    t = time.perf_counter(); c._calc_input_control(x); dt = time.perf_counter() - t
    tm = c.engine.timings()
    rows.append((dt * 1e6, tm["last_step_ms"] * 1e3, tm["last_rollout_ms"] * 1e3, tm["last_update_ms"] * 1e3, tm["last_passes"]))
r = np.median(np.array(rows), axis=0)
print("with events: host %.1f us, device step %.1f us = rollout (strict passes + round trips) %.1f + update kernel %.1f; passes %d" % tuple(r))
