import os, sys; sys.path[:0]=[os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]
import numpy as np, torch
from golden_util import Golden
from gpu_util import engine_from_spec
from oracle import mppi_oracle as orc
g = Golden("diffdrive_pe0.05")
for nin in (3,5):
    mlp = orc.make_mlp(seed=0, out_scale=0.01, n_hidden=2, n_in=nin)
    sp = orc.diffdrive_spec(K=65536, T=30, param_exploration=0.05, cost_mode="sum", waypoint_mode="frozen", model="diffdrive_mlp", mlp=mlp)
    sp.temperature = 2.0
    eng = engine_from_spec(sp, g.path)
    eng.set_mlp([mlp["W%d"%i] for i in range(4)],[mlp["b%d"%i] for i in range(4)])
    x0=np.array([0.4,0.3,0.5])
    for i in range(3): eng.step(x0, None, 7, i)
    eng.set_timing(True)
    r=[];u=[]
    for i in range(10):
        eng.step(x0, None, 7, 10+i); t=eng.timings(); r.append(t['last_rollout_ms']); u.append(t['last_update_ms'])
    print("n_in", nin, "rollout ms", np.median(r), "update (K2) ms", np.median(u))
    eng.close()
